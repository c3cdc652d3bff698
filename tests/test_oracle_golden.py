"""CPU: the oracle restatement reproduces the committed reference outputs (tests/golden/*.pt, produced by
oracle/make_golden.py from the UNMODIFIED reference)."""
import os

import pytest
import torch

from oracle import unet_oracle as UO, vae_oracle as VO, samplers_oracle as SO
from oracle.make_golden import analytic_model, _SchedModel, synth_inputs


def test_unet_tiny_matches_reference_fixture(gold_dir):
    g = torch.load(os.path.join(gold_dir, 'unet_tiny.pt'))
    cfg = UO.UNetConfig(**{**g['cfg'], 'dim_mult': tuple(g['cfg']['dim_mult']), 'attn_scales': tuple(g['cfg']['attn_scales'])})
    W = UO.make_weights(UO.param_specs(cfg), seed=g['wseed'])
    x, c, uc = synth_inputs(g['F'], g['h'], g['w'])
    taps = {}
    out = UO.unet_forward(W, cfg, x, torch.tensor([g['t']]), c, taps)
    assert torch.allclose(out, g['eps_cond'], rtol=0, atol=2e-5)
    assert torch.allclose(UO.unet_forward(W, cfg, x, torch.tensor([g['t']]), uc), g['eps_uncond'], rtol=0, atol=2e-5)
    ntap = 0
    for k, v in g.items():
        if k.startswith('tap:'):
            assert torch.allclose(taps[k[4:]].half().float(), v.float(), rtol=2e-3, atol=2e-3), k
            ntap += 1
    assert ntap >= 10


def test_param_specs_count_public_config():
    specs = UO.param_specs(UO.UNetConfig())
    assert len(specs) == 1480                                   # SURVEY.md appendix D
    n = sum(int(torch.tensor(s).prod()) for s in specs.values())
    assert abs(n / 1e6 - 1411.23) < 0.5                         # 1.41 B parameters


def test_vae_decode_matches_reference_fixture(gold_dir):
    g = torch.load(os.path.join(gold_dir, 'vae_decode.pt'))
    cfg = VO.VAEConfig()
    W = UO.make_weights(VO.decoder_param_specs(cfg), seed=g['wseed'])
    z = torch.randn(g['z_shape'], generator=torch.Generator('cpu').manual_seed(g['z_seed'])) * g['z_scale']
    out = VO.vae_decode(W, cfg, z)
    assert torch.allclose(out, g['out'], rtol=0, atol=1e-4)


@pytest.mark.parametrize('key,fn,S,scale', [
    ('ddim_gaussian_S50_g17.0', SO.ddim_gaussian_sample, 50, 17.0),
    ('ddim_gaussian_S20_g7.5', SO.ddim_gaussian_sample, 20, 7.5),
    ('ddim_gaussian_S7_g1.0', SO.ddim_gaussian_sample, 7, 1.0),
    ('ddim_S50_g17.0', SO.ddim_sample, 50, 17.0),
    ('ddim_S20_g7.5', SO.ddim_sample, 20, 7.5),
    ('ddim_S7_g1.0', SO.ddim_sample, 7, 1.0),
    ('unipc_S30_g17.0', SO.unipc_sample, 30, 17.0),
    ('unipc_S12_g7.5', SO.unipc_sample, 12, 7.5),
    ('unipc_S5_g1.0', SO.unipc_sample, 5, 1.0),
])
def test_sampler_trajectories_match_reference_fixture(gold_dir, key, fn, S, scale):
    g = torch.load(os.path.join(gold_dir, 'samplers.pt'))
    betas = SO.linear_sd_betas()
    x = torch.randn(g['shape'], generator=torch.Generator('cpu').manual_seed(g['x_seed']))
    c = torch.full((1, 77, 8), g['c_val'])
    uc = torch.full((1, 77, 8), g['uc_val'])
    torch.manual_seed(7)
    out = fn(_SchedModel(betas), betas, x, S, c, uc, scale)
    assert torch.allclose(out, g[key], rtol=0, atol=1e-6), (out - g[key]).abs().max()


def test_gaussian_cfg_guides_only_first_half_of_channels():
    """SURVEY.md appendix C: cond = 1, uncond = 0, g = 17 -> [17, 17, 1, 1]."""
    y = torch.ones(1, 4, 2, 2, 2)
    u = torch.zeros(1, 4, 2, 2, 2)
    out = SO.gaussian_cfg(y, u, 17.0)
    assert out[0, :, 0, 0, 0].tolist() == [17.0, 17.0, 1.0, 1.0]


def test_ddim_timestep_grids():
    ts, stride = SO.gaussian_timesteps(1000, 50)
    assert ts[0] == 981 and ts[-1] == 1 and stride == 20 and len(ts) == 50
    dts, *_ = SO.ddim_schedule(torch.cumprod(1 - SO.linear_sd_betas(), 0), 50)
    assert dts[0] == 1 and dts[-1] == 981


def test_oracle_unet_live_against_reference(gold_dir):
    """B = 2 with two different timesteps: oracle vs the reference UNetSD's output (tests/golden/unet_tiny_b2.pt)."""
    g = torch.load(os.path.join(gold_dir, 'unet_tiny_b2.pt'))
    cfg = UO.UNetConfig(dim=64)
    W = UO.make_weights(UO.param_specs(cfg), seed=g['wseed'])
    gen = torch.Generator().manual_seed(g['xy_seed'])
    x = torch.randn(g['x_shape'], generator=gen)
    y = torch.randn(g['y_shape'], generator=gen)
    assert torch.allclose(UO.unet_forward(W, cfg, x, g['t'], y), g['out'], rtol=0, atol=3e-5)


# ---------------------------------------------------------------------------------------- VideoCrafter (SURVEY.md 8 a19-a20)
from oracle import vc_oracle as VC  # noqa: E402


def _vc_inputs(g):
    B, _, T, h, w = g['shape']
    x = torch.randn(g['shape'], generator=torch.Generator('cpu').manual_seed(g['x_seed']))
    ctx = torch.randn((B, g['L'], g['cfg']['context_dim']), generator=torch.Generator('cpu').manual_seed(g['ctx_seed']))
    return x, ctx


@pytest.mark.parametrize('name', ['vc_unet_tiny', 'vc_unet_full'])
def test_vc_unet_matches_reference_fixture(gold_dir, name):
    g = torch.load(os.path.join(gold_dir, name + '.pt'))
    cfg = VC.VCConfig(**g['cfg'])
    W = UO.make_weights(VC.vc_param_specs(cfg), seed=g['wseed'])
    x, ctx = _vc_inputs(g)
    out = VC.vc_unet_forward(W, cfg, x, g['t'], ctx)
    assert torch.allclose(out, g['out'], rtol=0, atol=2e-5)


def test_vc_param_specs_count_public_config():
    specs = VC.vc_param_specs(VC.VCConfig())
    n = sum(int(torch.tensor(s).prod()) for s in specs.values())
    assert len(specs) == 974 and abs(n / 1e6 - 958.9) < 0.1      # SURVEY.md 8 a19: 958.9 M parameters


@pytest.mark.parametrize('S,scale,eta', [(50, 15.0, 0.0), (20, 7.5, 0.0), (10, 3.0, 0.5)])
def test_vc_ddim_matches_reference_fixture(gold_dir, S, scale, eta):
    g = torch.load(os.path.join(gold_dir, 'vc_ddim.pt'))
    x = torch.randn(g['shape'], generator=torch.Generator('cpu').manual_seed(g['x_seed']))
    c = torch.full((2, 77, 8), g['c_val'])
    uc = torch.full((2, 77, 8), g['uc_val'])
    o = VC.vc_ddim_sample(lambda xx, t, cc: analytic_model(xx, t, cc), SO.linear_sd_betas(), x, S, c, uc, scale, eta=eta,
                          noise_gen=torch.Generator('cpu').manual_seed(11))
    assert torch.allclose(o, g[f'S{S}_g{scale}_eta{eta}'], rtol=0, atol=1e-6)


def test_vae_encode_matches_reference_fixture(gold_dir):
    g = torch.load(os.path.join(gold_dir, 'vae_encode.pt'))
    cfg = VO.VAEConfig()
    W = UO.make_weights(VO.encoder_param_specs(cfg), seed=g['wseed'])
    x = torch.rand(g['x_shape'], generator=torch.Generator('cpu').manual_seed(g['x_seed'])) * 2 - 1
    mom = VO.vae_encode_moments(W, cfg, x)
    assert torch.allclose(mom[:, :4], g['mean'], rtol=0, atol=1e-5)
    assert torch.allclose(torch.clamp(mom[:, 4:], -30.0, 20.0), g['logvar'], rtol=0, atol=1e-5)


def test_unet_125_frames_matches_reference_fixture(gold_dir):
    """Config 4's frame count through the temporal modules (narrow net, B = 2): oracle vs the reference output."""
    g = torch.load(os.path.join(gold_dir, 'unet_f125.pt'))
    cfg = UO.UNetConfig(dim=64)
    W = UO.make_weights(UO.param_specs(cfg), seed=g['wseed'])
    x, c, uc = synth_inputs(g['F'], g['h'], g['w'])
    x = torch.cat([x, x.flip(2) * 0.5], 0)
    out = UO.unet_forward(W, cfg, x, g['t'], torch.cat([c, uc], 0))
    assert torch.allclose(out, g['eps'].float(), rtol=0, atol=2e-5)


def test_full_size_fixtures_are_consistent(gold_dir):
    """The full-model fixtures at BASELINE's shapes (config 2 / 3 / 5) are too expensive to re-derive in the CPU suite
    (make_golden.py asserted oracle == reference when it wrote them); check their shapes and that the single-step latents
    follow from the stored eps through the pinned scheduler restatement (DDIM_Gaussian: no model call needed)."""
    g = torch.load(os.path.join(gold_dir, 'unet_cfg2.pt'))
    assert (g['F'], g['h'], g['w']) == (24, 32, 32) and g['eps_cond'].shape == (1, 4, 24, 32, 32)
    x, c, uc = synth_inputs(24, 32, 32)
    calls = []

    def model(xx, tt, cc):
        calls.append(1)
        if len(calls) > 2:
            raise StopIteration
        return g['eps_cond'] if len(calls) == 1 else g['eps_uncond']
    tr = []
    try:
        SO.ddim_gaussian_sample(model, SO.linear_sd_betas(), x, 50, c, uc, 17.0, trace=tr)
    except StopIteration:
        pass
    s = g['x1_stride']                        # the latents after one update are stored as every s-th element
    assert torch.allclose(tr[0].reshape(-1)[::s], g['ddim_gaussian_x1'], rtol=0, atol=1e-6)
    for k in ('ddim_x1', 'unipc_x1'):
        assert g[k].shape == x.reshape(-1)[::s].shape and torch.isfinite(g[k]).all()
    g3 = torch.load(os.path.join(gold_dir, 'unet_cfg3_slice.pt'))
    assert g3['eps'].shape == (1, 4, 2, 72, 128)
    g5 = torch.load(os.path.join(gold_dir, 'vc_unet_cfg5.pt'))
    assert tuple(g5['out'].shape) == (1, 4, 16, 32, 32)
