"""CPU: the nn.Module mirrors expose the reference's state_dict / module tree (load_state_dict(strict=True), LoRA
name matching) and schedule buffers -- checked against the oracle's parameter table (itself pinned against the
reference) and against the reference classes' own layout, stored in tests/golden."""
import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import unet_oracle as UO, vae_oracle as VO
from oracle import samplers_oracle as SO
from t2v_b200.modules import UNetSD, AutoencoderKL
from t2v_b200.pipeline import VAE_DDCONFIG, linear_sd_betas


def test_unet_state_dict_layout_tiny():
    cfg = UO.UNetConfig(dim=64)
    net = UNetSD(dim=64)
    specs = UO.param_specs(cfg)
    sd = net.state_dict()
    assert {k: tuple(v.shape) for k, v in sd.items()} == {k: tuple(v) for k, v in specs.items()}
    net.load_state_dict(UO.make_weights(specs, seed=1), strict=True)
    with pytest.raises(RuntimeError):
        bad = dict(UO.make_weights(specs, seed=1))
        bad['not.a.key'] = torch.zeros(1)
        net.load_state_dict(bad, strict=True)


def test_unet_leaf_types_for_lora_and_typo_key():
    net = UNetSD(dim=64)
    mods = dict(net.named_modules())
    assert isinstance(mods['input_blocks.1.0.in_layers.2'], nn.Conv2d)
    assert isinstance(mods['input_blocks.1.0.temopral_conv.conv1.2'], nn.Conv3d)          # sic
    assert isinstance(mods['input_blocks.1.0.temopral_conv.conv2.3'], nn.Conv3d)
    assert isinstance(mods['input_blocks.1.1.transformer_blocks.0.attn2.to_k'], nn.Linear)
    assert isinstance(mods['input_blocks.1.2.proj_in'], nn.Conv1d)
    assert isinstance(mods['input_blocks.1.1.transformer_blocks.0.norm1'], nn.LayerNorm)
    assert isinstance(mods['input_blocks.1.1.norm'], nn.GroupNorm)
    assert mods['input_blocks.0.1.proj_in'].weight.shape == (512, 64, 1)                     # stem TT: 8 heads x 64
    # weights stay re-assignable Parameters (stable_lora/scripts/lora_processor.py:236-242)
    lin = mods['input_blocks.1.1.transformer_blocks.0.attn2.to_k']
    lin.weight = nn.Parameter(lin.weight.detach() * 2)


def test_vae_state_dict_layout():
    v = AutoencoderKL(VAE_DDCONFIG, 4)
    sd = {k: tuple(t.shape) for k, t in v.state_dict().items()}
    dec = VO.decoder_param_specs(VO.VAEConfig())
    for k, s in dec.items():
        assert sd[k] == tuple(s), k
    assert len(sd) == 248 and 'encoder.conv_in.weight' in sd and 'quant_conv.weight' in sd


def test_schedule_buffers_match_oracle():
    net = UNetSD(dim=64)
    betas = linear_sd_betas()
    assert torch.equal(betas, SO.linear_sd_betas())
    net.register_schedule(given_betas=betas.numpy())
    acp = torch.cumprod(1 - betas, 0)
    assert torch.equal(net.alphas_cumprod, acp.to(torch.float32))
    assert net.num_timesteps == 1000 and net.parameterization == 'eps'
    assert torch.equal(net.alphas_cumprod_prev[1:], acp[:-1].to(torch.float32)) and net.alphas_cumprod_prev[0] == 1


def test_cpu_forward_is_refused():
    net = UNetSD(dim=64)
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    with pytest.raises(RuntimeError):
        net(torch.zeros(1, 4, 2, 8, 8), torch.tensor([1]), torch.zeros(1, 77, 1024))


def test_mirror_against_reference_classes(gold_dir):
    """State-dict shapes and Linear / Conv classes of the mirrors vs the reference's UNetSD (dim 64) and AutoencoderKL
    (tests/golden/module_tree.pt, written by oracle/make_golden.py from the reference classes)."""
    import os
    ref = torch.load(os.path.join(gold_dir, 'module_tree.pt'))
    mine = UNetSD(dim=64)
    assert ref['unet_dim64']['state_dict'] == {k: tuple(v.shape) for k, v in mine.state_dict().items()}
    kinds = ('Linear', 'Conv1d', 'Conv2d', 'Conv3d')
    mt = {n: type(x).__name__ for n, x in mine.named_modules() if type(x).__name__ in kinds}
    assert ref['unet_dim64']['modules'] == mt
    mv = AutoencoderKL(VAE_DDCONFIG, 4)
    assert ref['vae']['state_dict'] == {k: tuple(v.shape) for k, v in mv.state_dict().items()}


# ---------------------------------------------------------------------------------------- VideoCrafter mirrors
def test_videocrafter_unet_state_dict_layout():
    from oracle import vc_oracle as VC
    from t2v_b200.modules import UNetModel
    for kw, cfg in ((dict(model_channels=64, context_dim=48, temporal_length=4),
                     VC.VCConfig(model_channels=64, context_dim=48, temporal_length=4)), (dict(), VC.VCConfig())):
        if kw:
            net = UNetModel(**kw)
        else:
            with torch.device('meta'):             # 958.9 M parameters: shapes only (no allocation / random init on the CPU)
                net = UNetModel()
        specs = VC.vc_param_specs(cfg)
        assert {k: tuple(v.shape) for k, v in net.state_dict().items()} == {k: tuple(v) for k, v in specs.items()}
    mods = dict(net.named_modules())
    assert isinstance(mods['input_blocks.1.0.in_layers.2'], nn.Conv3d)                                   # (1,3,3) kernels
    assert mods['input_blocks.1.0.in_layers.2'].weight.shape == (320, 320, 1, 3, 3)
    assert isinstance(mods['input_blocks.1.1.transformer_blocks.0.norm5'], nn.LayerNorm)
    assert isinstance(mods['input_blocks.1.1.transformer_blocks.0.attn2.to_k'], nn.Linear)
    assert mods['input_blocks.1.1.transformer_blocks.0.attn2.to_k'].weight.shape == (320, 768)
    assert mods['input_blocks.1.1.transformer_blocks.0.attn1_tmp.relative_position_k'].embeddings_table.shape == (33, 40)
    with pytest.raises(NotImplementedError):
        UNetModel(use_scale_shift_norm=True)


def test_videocrafter_latent_diffusion_layout_and_schedule():
    from t2v_b200.videocrafter import LatentDiffusion, DDIMSampler, make_model_input_shape
    m = LatentDiffusion(unet_config=dict(model_channels=64, context_dim=48, temporal_length=4), image_size=[8, 8], video_length=4)
    keys = set(m.state_dict())
    assert any(k.startswith('model.diffusion_model.input_blocks.') for k in keys)
    assert 'first_stage_model.encoder.conv_in.weight' in keys and 'first_stage_model.post_quant_conv.bias' in keys
    assert make_model_input_shape(m, 2) == [2, 4, 4, 8, 8] and make_model_input_shape(m, 1, T=6) == [1, 4, 6, 8, 8]
    assert torch.equal(m.betas, SO.linear_sd_betas().to(torch.float32)) and m.num_timesteps == 1000
    smp = DDIMSampler(m)
    smp.make_schedule(50, ddim_eta=0.0)
    ts, alphas, alphas_prev, sigmas = SO.ddim_schedule(torch.cumprod(1 - SO.linear_sd_betas(), 0), 50, 0.0)
    assert (smp.ddim_timesteps == ts).all() and abs(float(smp.ddim_alphas[7]) - float(alphas[7])) < 1e-7
    with pytest.raises(RuntimeError):
        m.get_learned_conditioning(['text'])


@pytest.mark.parametrize('strength,steps', [(0.6, 20), (0.25, 30), (1.0, 10)])
def test_vid2vid_entry_noise_matches_reference_fixture(gold_dir, strength, steps):
    """encode_latent's three back ends (samplers_common.py:123-145) are host-side torch arithmetic: checked on CPU against
    the reference's outputs (tests/golden/vid2vid_encode.pt, written by oracle/make_golden.py)."""
    import os
    from t2v_b200 import samplers as M
    gd = torch.load(os.path.join(gold_dir, 'vid2vid_encode.pt'))
    g = torch.Generator().manual_seed(gd['lat_noise_seed'])
    lat = torch.randn(gd['shape'], generator=g)
    noise = torch.randn(gd['shape'], generator=g)
    ref = gd[f's{strength}_n{steps}']
    betas = linear_sd_betas()
    net = UNetSD(dim=64)
    net.register_schedule(given_betas=betas.numpy())
    n = int(strength * steps)
    if ref['ddim'] is not None:
        md = M.DDIMSampler(net, device=torch.device('cpu'))
        md.make_schedule(steps)
        # the reference returns fp64 here (numpy schedule) and encode_latent casts back to the latent dtype (:136)
        assert torch.allclose(md.stochastic_encode(lat, torch.tensor([n]), noise=noise), ref['ddim'].float(), rtol=0, atol=1e-6)
    assert torch.equal(M.UniPCSampler(net).unipc_encode(lat, torch.device('cpu'), strength, steps, noise=noise), ref['unipc'])
    mg = M.GaussianDiffusion(net, betas)
    assert torch.equal(mg.add_noise(lat, noise, mg.get_time_steps(n, 1)[0]), ref['gauss'])


@pytest.mark.parametrize('frames,i_frames,spec', [
    (8, 4, '0:(t/max_i_f), "max_i_f":(1)'), (24, 8, '0:(t/max_i_f), "max_i_f":(1)'), (6, 4, '0:(0.25), 3:(1.0)'),
    (10, 3, '0:(0), 4:(0.5), "max_f":(1)'), (12, 6, '0:(sin(t/max_f)), 9:(0.2)'),
    (8, 4, '0:(t/max_i_f), "max_i_f":(1*1)'), (16, 5, '0:(0.1+t/max_f), 11:(t*t/(max_f*max_f))')])
def test_inpainting_weight_schedule_matches_reference(gold_dir, frames, i_frames, spec):
    """T2VAnimKeys (t2v_helpers/key_frames.py:9-95) restated without numexpr / pandas: same per-frame weights, including the
    reference's 'expression sticks until the next numeric key' behaviour."""
    from types import SimpleNamespace as NS
    from t2v_b200.key_frames import T2VAnimKeys
    got = T2VAnimKeys(NS(max_frames=frames, inpainting_weights=spec), 7, i_frames).inpainting_weights_series
    expected = {
        (8, 4, '0:(t/max_i_f), "max_i_f":(1)'): [0, 1 / 3, 2 / 3, 1, 1, 1, 1, 1],
        (6, 4, '0:(0.25), 3:(1.0)'): [0.25, 0.5, 0.75, 1, 1, 1],
    }.get((frames, i_frames, spec))
    if expected is not None:
        assert np.allclose(got, expected)
    # the unmodified reference class's weights for the same spec (tests/golden/key_frames.json, oracle/make_golden.py)
    import json
    import os
    with open(os.path.join(gold_dir, 'key_frames.json')) as f:
        ref = [c['weights'] for c in json.load(f)['cases'] if (c['frames'], c['i_frames'], c['spec']) == (frames, i_frames, spec)]
    assert len(ref) == 1
    if ref[0] is None:
        # numeric keys: the reference stores the STRING into a float64 Series (key_frames.py:38), which pandas >= 3
        # rejects -- the unmodified reference could not run those specs when the fixture was written; the
        # expression-valued specs are compared
        assert any(ch.isdigit() for ch in spec)
        return
    assert np.allclose(got, np.asarray(ref[0], dtype=np.float64), rtol=0, atol=1e-12)


def test_stable_lora_processor_walk_and_flags_on_cpu():
    """Host side of the LoRA hot-merge (stable_lora/stable_utils/lora_processor.py:202-246): which `<name>.lora_A/B` pairs reach
    the device-side merge, with which flags -- on a CPU mirror whose `lora_merge` / `lora_clear` are replaced by recorders."""
    from t2v_b200.modules import UNetSD
    from t2v_b200.lora import StableLoraProcessor
    with torch.device('meta'):
        net = UNetSD(dim=64)
    calls = []
    net.lora_merge = lambda name, A, B, alpha, temporal_mean=False: calls.append((name, tuple(A.shape), tuple(B.shape), alpha, temporal_mean))
    cleared = []
    net.lora_clear = lambda: cleared.append(True)
    r = 4
    lin, conv2, conv3, proj = ('input_blocks.1.1.transformer_blocks.0.attn1.to_q', 'input_blocks.1.0.in_layers.2',
                               'input_blocks.1.0.temopral_conv.conv1.2', 'input_blocks.1.1.proj_in')
    lora = {lin + '.lora_A': torch.zeros(r, 64), lin + '.lora_B': torch.zeros(64, r),
            conv2 + '.lora_A': torch.zeros(r, 64 * 9), conv2 + '.lora_B': torch.zeros(64, r),
            conv3 + '.lora_A': torch.zeros(r, 64 * 9), conv3 + '.lora_B': torch.zeros(64, r),
            proj + '.lora_A': torch.zeros(r, 64, 1), proj + '.lora_B': torch.zeros(64, r, 1),       # Conv1d-style tensors get squeezed (:222-223)
            'not.a.module.lora_A': torch.zeros(r, 8), 'not.a.module.lora_B': torch.zeros(8, r)}
    p = StableLoraProcessor()
    assert p.process_lora(net, [lora], lora_alpha=0.5) == 4
    got = {c[0]: c for c in calls}
    assert got[lin + '.weight'][3:] == (0.5, False) and got[conv2 + '.weight'][4] is False
    assert got[conv3 + '.weight'][4] is True                                   # Conv3d (3,1,1): product averaged over the kernel axis
    assert got[proj + '.weight'][1] == (r, 64) and got[proj + '.weight'][2] == (64, r)
    calls.clear()
    assert p.process_lora(net, [lora], use_conv=False) == 2 and {c[0] for c in calls} == {lin + '.weight', proj + '.weight'}
    calls.clear()
    assert p.process_lora(net, [lora], use_time=False) == 3 and conv3 + '.weight' not in {c[0] for c in calls}
    assert p.process_lora(net, [], undo_merge=True) == 0 and cleared == [True] and p.previous is None
    with pytest.raises(NotImplementedError):
        p.process_lora(net, [lora], use_bias=True)
    with pytest.raises(TypeError):
        p.process_lora(nn.Linear(2, 2), [lora])


def test_default_video_encoder_returns_a_data_url_with_exact_frames():
    """process_modelscope returns data-URL strings like the reference (process_modelscope.py:34).  Without ffmpeg the default
    encoder wraps the frames in an uncompressed RIFF AVI: decode the URL again and compare the pixels."""
    import base64
    import struct
    import numpy as np
    from t2v_b200 import video_encode as VE
    rng = np.random.default_rng(0)
    frames = [rng.integers(0, 256, size=(6, 5, 3), dtype=np.uint8) for _ in range(3)]       # odd width: rows are padded to 4 bytes
    raw = VE._avi_bytes(frames, 8.0)
    assert raw[:4] == b'RIFF' and raw[8:12] == b'AVI ' and struct.unpack('<I', raw[4:8])[0] == len(raw) - 8
    url = VE.default_video_encoder(frames)
    assert url.startswith('data:video/mp4;base64,') or url.startswith('data:video/avi;base64,')
    if url.startswith('data:video/avi'):
        assert base64.b64decode(url.split(',', 1)[1]) == VE._avi_bytes(frames, 15.0)
    # frame payloads: '00db' chunks, bottom-up rows of w*3 bytes padded to a multiple of 4
    pos, got = raw.index(b'movi') + 4, []
    for _ in frames:
        assert raw[pos:pos + 4] == b'00db'
        n = struct.unpack('<I', raw[pos + 4:pos + 8])[0]
        rows = np.frombuffer(raw[pos + 8:pos + 8 + n], dtype=np.uint8).reshape(6, 16)[:, :15].reshape(6, 5, 3)
        got.append(rows[::-1])
        pos += 8 + n + (n & 1)
    assert all(np.array_equal(a, b) for a, b in zip(got, frames))
