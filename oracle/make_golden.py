"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.pt by executing the UNMODIFIED reference
(/root/reference, imported through oracle/ref_shim.py) on CPU fp32, and cross-checks the oracle
restatement against it while doing so.  Run in the build container (the reference does not exist
on the GPU box):

    python oracle/make_golden.py            # writes tests/golden/*.pt, prints oracle-vs-reference errors
    python oracle/make_golden.py unet_cfg2  # only the named fixtures

Fixtures hold inputs' seeds + reference OUTPUTS only; weights are regenerated from seeds by
oracle.unet_oracle.make_weights (bit-identical on any host with the same torch build).
"""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_shim                                   # noqa: E402
from oracle import unet_oracle as UO                          # noqa: E402
from oracle import vae_oracle as VO                           # noqa: E402
from oracle import samplers_oracle as SO                      # noqa: E402
from oracle import vc_oracle as VC                            # noqa: E402

GOLD = os.path.join(ROOT, 'tests', 'golden')
# fixture files stay under 1 MB: the full-size single-step fixture keeps every X1_STRIDE-th element of its three
# after-one-update latents (7 is odd, so the sample walks through every row, column, frame and channel)
X1_STRIDE = 7


def build_ref_unet(m, cfg: UO.UNetConfig):
    return m.UNetSD(in_dim=cfg.in_dim, dim=cfg.dim, y_dim=768, context_dim=cfg.context_dim,
                    out_dim=cfg.out_dim, dim_mult=list(cfg.dim_mult), num_heads=cfg.num_heads,
                    head_dim=cfg.head_dim, num_res_blocks=cfg.num_res_blocks,
                    attn_scales=list(cfg.attn_scales), dropout=0.1, temporal_attention=True).eval()


def synth_inputs(F, h, w, L=77, ctx_dim=1024, seed=123):
    """x_T exactly as samplers_common.py:118-119 (CPU generator seeded per run); cond/uncond from seed 2."""
    g = torch.Generator('cpu').manual_seed(seed)
    x = torch.randn((1, 4, F, h, w), generator=g)
    g2 = torch.Generator('cpu').manual_seed(2)
    c = torch.randn(1, L, ctx_dim, generator=g2)
    uc = torch.randn(1, L, ctx_dim, generator=g2)
    return x, c, uc


def gold_unet(m, name, cfg, F, h, w, wseed, keep_taps):
    torch.manual_seed(0)
    net = build_ref_unet(m, cfg)
    specs = UO.param_specs(cfg)
    sd = net.state_dict()
    assert set(sd) == set(specs), (set(sd) ^ set(specs))
    for k in sd:
        assert tuple(sd[k].shape) == specs[k], k
    W = UO.make_weights(specs, seed=wseed)
    net.load_state_dict(W, strict=True)
    x, c, uc = synth_inputs(F, h, w, ctx_dim=cfg.context_dim)
    t = torch.tensor([981])
    ref_taps = {}
    hooks = []
    if keep_taps:
        for mname, mod in net.named_modules():
            if mname in keep_taps:
                hooks.append(mod.register_forward_hook(
                    lambda mod_, inp, out, n=mname: ref_taps.__setitem__(n, out.detach().clone())))
    t0 = time.time()
    with torch.no_grad():
        eps_c = net(x, t, c)
        for hk in hooks:
            hk.remove()
        eps_u = net(x, t, uc)
    dt = time.time() - t0
    taps = {}
    o_c = UO.unet_forward(W, cfg, x, t, c, taps)
    o_u = UO.unet_forward(W, cfg, x, t, uc)
    err = max((o_c - eps_c).abs().max().item(), (o_u - eps_u).abs().max().item())
    print(f'[{name}] reference 2 forwards {dt:.1f}s; oracle-vs-reference max|d| = {err:.3e} '
          f'(ref absmax {eps_c.abs().max().item():.3f})')
    assert err < 2e-4
    out = {'cfg': cfg.__dict__, 'F': F, 'h': h, 'w': w, 'wseed': wseed, 'x_seed': 123, 'ctx_seed': 2,
           't': 981, 'eps_cond': eps_c, 'eps_uncond': eps_u}
    for n, v in ref_taps.items():
        # 5-D temporal modules are hooked in b c f h w; store everything as (b f) c h w
        if v.dim() == 5:
            v = v.permute(0, 2, 1, 3, 4).reshape(-1, v.shape[1], v.shape[3], v.shape[4])
        d = (taps[n] - v).abs().max().item()
        assert d < 2e-4, (n, d)
        out['tap:' + n] = v.half()
    # one sampler step of each scheduler from x_T, produced by the reference sampler classes: the
    # denoiser is wrapped so that the latent handed to the (n+1)-th model call -- i.e. the state after
    # the first update -- is captured and the run is then aborted.
    smp = ref_shim.load_samplers()
    betas = SO.linear_sd_betas()
    net.register_schedule(given_betas=betas.numpy())
    smp.SamplerBase('x', None).register_buffers_to_model(net, betas, torch.device('cpu'))
    from samplers.ddim.gaussian_sampler import GaussianDiffusion
    from samplers.ddim.sampler import DDIMSampler
    from samplers.uni_pc.sampler import UniPCSampler
    import samplers.uni_pc.sampler as ups
    ups.UniPCSampler.register_buffer = lambda self, nm, attr: setattr(self, nm, attr)   # see gold_samplers

    class _Stop(Exception):
        pass

    class Wrapped:
        def __init__(self, stop_at):
            self.calls, self.stop_at = [], stop_at
            for a_ in ('device', 'betas', 'alphas_cumprod', 'alphas_cumprod_prev', 'num_timesteps',
                       'parameterization'):
                setattr(self, a_, getattr(net, a_))

        def __call__(self, xx, tt, cc):
            self.calls.append(xx.clone())
            if len(self.calls) == self.stop_at:
                raise _Stop()
            return net(xx, tt, cc)

    def first_update(run, stop_at):
        wm = Wrapped(stop_at)
        try:
            run(wm)
        except _Stop:
            pass
        return wm.calls[-1]

    S = 50
    out['ddim_gaussian_x1'] = first_update(
        lambda wm: GaussianDiffusion(wm, betas).sample(x_T=x, S=S, conditioning=c, unconditional_conditioning=uc,
                                                       unconditional_guidance_scale=17.0, eta=0.0), 3)
    out['ddim_x1'] = first_update(
        lambda wm: DDIMSampler(wm, device=torch.device('cpu')).sample(
            S=S, batch_size=1, shape=tuple(x.shape), conditioning=c, x_T=x, unconditional_guidance_scale=17.0,
            unconditional_conditioning=uc, eta=0.0), 3)
    out['unipc_x1'] = first_update(
        lambda wm: UniPCSampler(wm).sample(S=30, batch_size=1, shape=tuple(x.shape), conditioning=c, x_T=x,
                                           unconditional_guidance_scale=17.0, unconditional_conditioning=uc,
                                           strength=None), 5)
    # the oracle samplers driven by the oracle UNet must hand the same latent to the same model call
    # (for UniPC the 5th call receives the *predictor* output of the 2nd update, uni_pc.py:630-645)
    class OWrapped:
        def __init__(self, stop_at):
            self.calls, self.stop_at = [], stop_at

        def __call__(self, xx, tt, cc):
            self.calls.append(xx.clone())
            if len(self.calls) == self.stop_at:
                raise _Stop()
            return UO.unet_forward(W, cfg, xx, tt, cc)

    for key, stop_at, fn in (
            ('ddim_gaussian_x1', 3, lambda om: SO.ddim_gaussian_sample(om, betas, x, S, c, uc, 17.0)),
            ('ddim_x1', 3, lambda om: SO.ddim_sample(om, betas, x, S, c, uc, 17.0)),
            ('unipc_x1', 5, lambda om: SO.unipc_sample(om, betas, x, 30, c, uc, 17.0))):
        om = OWrapped(stop_at)
        try:
            fn(om)
        except _Stop:
            pass
        d = (om.calls[-1] - out[key]).abs().max().item()
        print(f'[{name}] {key}: oracle-vs-reference max|d| = {d:.3e}')
        assert d < 5e-4, (key, d)
    torch.save(out, os.path.join(GOLD, name + '.pt'))
    return out



def gold_unet_step(m, name, cfg, F, h, w, wseed, unipc=True):
    """Full-size single-step gate at a BASELINE shape (config 2: 24 f x 32 x 32 latent): the reference module's eps for the
    cond / uncond branch at the first timestep and the latent after ONE update of each scheduler, produced by the reference
    sampler classes.  Reference forwards are memoised on (x, t, ctx) -- the first two model calls of DDIM_Gaussian and DDIM
    are the eps_cond / eps_uncond forwards themselves -- so the fixture costs 2 (+4 for UniPC) reference forwards."""
    torch.manual_seed(0)
    net = build_ref_unet(m, cfg)
    specs = UO.param_specs(cfg)
    W = UO.make_weights(specs, seed=wseed)
    net.load_state_dict(W, strict=True)
    x, c, uc = synth_inputs(F, h, w, ctx_dim=cfg.context_dim)
    memo = {}

    def ref_forward(xx, tt, cc):
        key = (float(tt.reshape(-1)[0]), float(cc.sum()), float(xx.double().sum()), float(xx.double().abs().sum()))
        if key not in memo:
            t0 = time.time()
            with torch.no_grad():
                memo[key] = net(xx, tt, cc)
            print(f'[{name}] reference forward t={key[0]:.1f} {time.time() - t0:.1f}s', flush=True)
        return memo[key]

    t = torch.tensor([981])
    eps_c = ref_forward(x, t, c)
    eps_u = ref_forward(x, t, uc)
    t0 = time.time()
    o_c = UO.unet_forward(W, cfg, x, t, c)
    err = (o_c - eps_c).abs().max().item()
    print(f'[{name}] oracle forward {time.time() - t0:.1f}s; oracle-vs-reference max|d| = {err:.3e} '
          f'(ref absmax {eps_c.abs().max().item():.3f})', flush=True)
    assert err < 2e-4
    out = {'cfg': cfg.__dict__, 'F': F, 'h': h, 'w': w, 'wseed': wseed, 'x_seed': 123, 'ctx_seed': 2, 't': 981,
           'eps_cond': eps_c, 'eps_uncond': eps_u}
    smp = ref_shim.load_samplers()
    betas = SO.linear_sd_betas()
    net.register_schedule(given_betas=betas.numpy())
    smp.SamplerBase('x', None).register_buffers_to_model(net, betas, torch.device('cpu'))
    from samplers.ddim.gaussian_sampler import GaussianDiffusion
    from samplers.ddim.sampler import DDIMSampler
    from samplers.uni_pc.sampler import UniPCSampler
    import samplers.uni_pc.sampler as ups
    ups.UniPCSampler.register_buffer = lambda self, nm, attr: setattr(self, nm, attr)

    class _Stop(Exception):
        pass

    class Wrapped:
        def __init__(self, stop_at):
            self.calls, self.stop_at = [], stop_at
            for a_ in ('device', 'betas', 'alphas_cumprod', 'alphas_cumprod_prev', 'num_timesteps', 'parameterization'):
                setattr(self, a_, getattr(net, a_))

        def __call__(self, xx, tt, cc):
            self.calls.append(xx.clone())
            if len(self.calls) == self.stop_at:
                raise _Stop()
            return ref_forward(xx, tt, cc)

    def first_update(run, stop_at):
        wm = Wrapped(stop_at)
        try:
            run(wm)
        except _Stop:
            pass
        return wm.calls[-1]

    S = 50
    out['ddim_gaussian_x1'] = first_update(
        lambda wm: GaussianDiffusion(wm, betas).sample(x_T=x, S=S, conditioning=c, unconditional_conditioning=uc,
                                                       unconditional_guidance_scale=17.0, eta=0.0), 3)
    out['ddim_x1'] = first_update(
        lambda wm: DDIMSampler(wm, device=torch.device('cpu')).sample(
            S=S, batch_size=1, shape=tuple(x.shape), conditioning=c, x_T=x, unconditional_guidance_scale=17.0,
            unconditional_conditioning=uc, eta=0.0), 3)
    if unipc:
        out['unipc_x1'] = first_update(
            lambda wm: UniPCSampler(wm).sample(S=30, batch_size=1, shape=tuple(x.shape), conditioning=c, x_T=x,
                                               unconditional_guidance_scale=17.0, unconditional_conditioning=uc,
                                               strength=None), 5)
    # the oracle samplers fed with the REFERENCE eps (memoised) must produce the same updates: pins the schedulers at this shape
    for key, stop_at, fn in (
            ('ddim_gaussian_x1', 3, lambda om: SO.ddim_gaussian_sample(om, betas, x, S, c, uc, 17.0)),
            ('ddim_x1', 3, lambda om: SO.ddim_sample(om, betas, x, S, c, uc, 17.0)),
            ('unipc_x1', 5, lambda om: SO.unipc_sample(om, betas, x, 30, c, uc, 17.0))):
        if key not in out:
            continue
        om = Wrapped(stop_at)
        try:
            fn(om)
        except _Stop:
            pass
        d = (om.calls[-1] - out[key]).abs().max().item()
        print(f'[{name}] {key}: oracle-sampler-vs-reference max|d| = {d:.3e}', flush=True)
        assert d < 5e-4, (key, d)
    for key in ('ddim_gaussian_x1', 'ddim_x1', 'unipc_x1'):
        if key in out:
            out[key] = out[key].reshape(-1)[::X1_STRIDE].clone()
    out['x1_stride'] = X1_STRIDE
    torch.save(out, os.path.join(GOLD, name + '.pt'))
    return out


def gold_unet_forward_only(m, name, cfg, F, h, w, wseed, B=1):
    """One reference forward (cond branch) at a shape that exercises a different kernel plan: config 3's S = 9216 spatial
    sequences (2 frames of 72 x 128 latent), or a 125-frame temporal path on a narrow net (config 4)."""
    torch.manual_seed(0)
    net = build_ref_unet(m, cfg)
    W = UO.make_weights(UO.param_specs(cfg), seed=wseed)
    net.load_state_dict(W, strict=True)
    x, c, uc = synth_inputs(F, h, w, ctx_dim=cfg.context_dim)
    if B == 2:
        x = torch.cat([x, x.flip(2) * 0.5], 0)
        c = torch.cat([c, uc], 0)
    t = torch.tensor([981, 37][:B])
    t0 = time.time()
    with torch.no_grad():
        eps = net(x, t, c)
    t1 = time.time()
    o = UO.unet_forward(W, cfg, x, t, c)
    err = (o - eps).abs().max().item()
    print(f'[{name}] reference {t1 - t0:.1f}s oracle {time.time() - t1:.1f}s; oracle-vs-reference max|d| = {err:.3e} '
          f'(ref absmax {eps.abs().max().item():.3f})', flush=True)
    assert err < 2e-4
    torch.save({'cfg': cfg.__dict__, 'F': F, 'h': h, 'w': w, 'B': B, 'wseed': wseed, 'x_seed': 123, 'ctx_seed': 2, 't': t,
                'eps': eps.half() if eps.numel() > (1 << 20) else eps}, os.path.join(GOLD, name + '.pt'))


class _SchedModel:
    """Stand-in denoiser exposing what the reference samplers read from the model
    (ddim/sampler.py:14,27-33; uni_pc/sampler.py:11-12; samplers_common.py:77-83)."""

    def __init__(self, betas):
        self.device = torch.device('cpu')
        self.betas = betas
        self.alphas_cumprod = torch.cumprod(1 - betas, dim=0)
        acp = self.alphas_cumprod.numpy()
        self.alphas_cumprod_prev = torch.tensor(np.append(1.0, acp[:-1]), dtype=torch.float32)
        self.num_timesteps = len(betas)
        self.parameterization = 'eps'

    def __call__(self, x, t, c):
        return analytic_model(x, t, c)


def analytic_model(x, t, c):
    """Cheap deterministic eps-model used to pin the schedulers without a UNet."""
    tt = t.float().view(-1, *((1,) * (x.ndim - 1))) / 1000.0
    bias = c.float().mean() if c is not None else 0.0
    ch = torch.arange(x.shape[1], dtype=x.dtype, device=x.device).view(1, -1, *((1,) * (x.ndim - 2)))
    return (torch.tanh(0.8 * x + 0.5 * tt + 0.1 * ch) * 0.9 + 0.3 * bias + 0.05 * torch.roll(x, 1, dims=2)).to(x.dtype)


def gold_samplers():
    ref_shim.load_samplers()
    from samplers.ddim.gaussian_sampler import GaussianDiffusion
    from samplers.ddim.sampler import DDIMSampler
    from samplers.uni_pc.sampler import UniPCSampler
    import samplers.uni_pc.sampler as ups
    betas = SO.linear_sd_betas()
    g = torch.Generator('cpu').manual_seed(123)
    x = torch.randn((1, 4, 5, 6, 7), generator=g)
    c = torch.full((1, 77, 8), 0.25)
    uc = torch.full((1, 77, 8), -0.5)
    model = _SchedModel(betas)
    out = {'x_seed': 123, 'shape': tuple(x.shape), 'c_val': 0.25, 'uc_val': -0.5}
    for S, scale in ((50, 17.0), (20, 7.5), (7, 1.0)):
        torch.manual_seed(7)
        r = GaussianDiffusion(model, betas).sample(x_T=x, S=S, conditioning=c, unconditional_conditioning=uc,
                                                   unconditional_guidance_scale=scale, eta=0.0)
        torch.manual_seed(7)
        o = SO.ddim_gaussian_sample(model, betas, x, S, c, uc, scale)
        print(f'[samplers] DDIM_Gaussian S={S} g={scale}: oracle-vs-reference max|d| = {(r - o).abs().max().item():.3e}')
        assert torch.allclose(r, o, rtol=0, atol=1e-6)
        out[f'ddim_gaussian_S{S}_g{scale}'] = r
        torch.manual_seed(7)
        r = DDIMSampler(model, device=torch.device('cpu')).sample(
            S=S, batch_size=1, shape=tuple(x.shape), conditioning=c, x_T=x,
            unconditional_guidance_scale=scale, unconditional_conditioning=uc, eta=0.0)
        torch.manual_seed(7)
        o = SO.ddim_sample(model, betas, x, S, c, uc, scale)
        print(f'[samplers] DDIM S={S} g={scale}: oracle-vs-reference max|d| = {(r - o).abs().max().item():.3e}')
        assert torch.allclose(r, o, rtol=0, atol=1e-6)
        out[f'ddim_S{S}_g{scale}'] = r
    # UniPCSampler.register_buffer hard-codes torch.device("cuda") (uni_pc/sampler.py:14-18): keep it on CPU here
    ups.UniPCSampler.register_buffer = lambda self, name, attr: setattr(self, name, attr)
    for S, scale in ((30, 17.0), (12, 7.5), (5, 1.0)):
        r = UniPCSampler(model).sample(S=S, batch_size=1, shape=tuple(x.shape), conditioning=c, x_T=x,
                                       unconditional_guidance_scale=scale, unconditional_conditioning=uc,
                                       strength=None)
        o = SO.unipc_sample(model, betas, x, S, c, uc, scale)
        print(f'[samplers] UniPC S={S} g={scale}: oracle-vs-reference max|d| = {(r - o).abs().max().item():.3e}')
        assert torch.allclose(r, o, rtol=0, atol=2e-5)
        out[f'unipc_S{S}_g{scale}'] = r
    # with eta > 0 (consumes the global RNG identically)
    torch.manual_seed(11)
    r = DDIMSampler(model, device=torch.device('cpu')).sample(
        S=10, batch_size=1, shape=tuple(x.shape), conditioning=c, x_T=x,
        unconditional_guidance_scale=3.0, unconditional_conditioning=uc, eta=0.5)
    torch.manual_seed(11)
    o = SO.ddim_sample(model, betas, x, 10, c, uc, 3.0, eta=0.5)
    assert torch.allclose(r, o, rtol=0, atol=1e-6)
    out['ddim_S10_g3.0_eta0.5_seed11'] = r
    torch.save(out, os.path.join(GOLD, 'samplers.pt'))


def gold_vae(m):
    cfg = VO.VAEConfig()
    ddconfig = {'double_z': True, 'z_channels': 4, 'resolution': 256, 'in_channels': 3, 'out_ch': 3, 'ch': 128,
                'ch_mult': [1, 2, 4, 4], 'num_res_blocks': 2, 'attn_resolutions': [], 'dropout': 0.0}
    torch.manual_seed(0)
    ae = m.AutoencoderKL(ddconfig, 4, None).eval()
    specs = VO.decoder_param_specs(cfg)
    sd = ae.state_dict()
    dec_keys = {k for k in sd if k.startswith('decoder.') or k.startswith('post_quant_conv.')}
    assert dec_keys == set(specs), dec_keys ^ set(specs)
    for k in specs:
        assert tuple(sd[k].shape) == specs[k], k
    W = UO.make_weights(specs, seed=3)
    sd.update(W)
    ae.load_state_dict(sd, strict=True)
    g = torch.Generator('cpu').manual_seed(5)
    z = torch.randn((2, 4, 8, 16), generator=g) / 0.18215 * 0.8
    with torch.no_grad():
        ref = ae.decode(z)
    o = VO.vae_decode(W, cfg, z)
    err = (o - ref).abs().max().item()
    print(f'[vae] oracle-vs-reference max|d| = {err:.3e} (ref absmax {ref.abs().max().item():.3f})')
    assert err < 1e-3 * max(1.0, ref.abs().max().item())
    torch.save({'wseed': 3, 'z_seed': 5, 'z_shape': (2, 4, 8, 16), 'z_scale': 0.8 / 0.18215, 'out': ref},
               os.path.join(GOLD, 'vae_decode.pt'))



def build_ref_vc_unet(cfg: VC.VCConfig):
    from videocrafter.lvdm.models.modules.openaimodel3d import UNetModel
    return UNetModel(image_size=32, in_channels=cfg.in_channels, out_channels=cfg.out_channels,
                     model_channels=cfg.model_channels, attention_resolutions=list(cfg.attention_resolutions),
                     num_res_blocks=cfg.num_res_blocks, channel_mult=list(cfg.channel_mult), num_heads=cfg.num_heads,
                     transformer_depth=1, context_dim=cfg.context_dim, use_checkpoint=False, legacy=False, kernel_size_t=1,
                     padding_t=0, temporal_length=cfg.temporal_length,
                     use_relative_position=cfg.use_relative_position).eval()


def gold_vc_unet(name, cfg: VC.VCConfig, B, T, h, w, L, wseed, half_out=False):
    """VideoCrafter UNetModel (SURVEY.md 8 a19): reference output on seeded inputs / weights; asserts the restatement."""
    torch.manual_seed(0)
    net = build_ref_vc_unet(cfg)
    specs = VC.vc_param_specs(cfg)
    sd = net.state_dict()
    assert set(sd) == set(specs), (set(sd) ^ set(specs))
    for k in sd:
        assert tuple(sd[k].shape) == specs[k], k
    W = UO.make_weights(specs, seed=wseed)
    net.load_state_dict(W, strict=True)
    g = torch.Generator('cpu').manual_seed(123)
    x = torch.randn((B, 4, T, h, w), generator=g)
    ctx = torch.randn((B, L, cfg.context_dim), generator=torch.Generator('cpu').manual_seed(2))
    t = torch.tensor([981, 37][:B])
    t0 = time.time()
    with torch.no_grad():
        ref = net(x, t, context=ctx)
    t1 = time.time()
    o = VC.vc_unet_forward(W, cfg, x, t, ctx)
    err = (o - ref).abs().max().item()
    print(f'[vc_unet:{name}] reference {t1 - t0:.1f}s; oracle-vs-reference max|d| = {err:.3e} '
          f'(ref absmax {ref.abs().max().item():.3f}), params {sum(v.numel() for v in W.values()) / 1e6:.2f} M')
    assert err <= 1e-5 * max(1.0, ref.abs().max().item())
    torch.save({'wseed': wseed, 'x_seed': 123, 'ctx_seed': 2, 'shape': (B, 4, T, h, w), 'L': L, 't': t, 'out': ref.half() if half_out else ref,
                'cfg': {'model_channels': cfg.model_channels, 'context_dim': cfg.context_dim,
                        'temporal_length': cfg.temporal_length}},
               os.path.join(GOLD, name + '.pt'))


def gold_vc_ddim():
    """lvdm/samplers/ddim.py DDIMSampler on the analytic eps-model (5-D latents, B = 2, with and without eta)."""
    ref_shim.install()
    from videocrafter.lvdm.samplers.ddim import DDIMSampler
    DDIMSampler.register_buffer = lambda self, name, attr: setattr(self, name, attr)    # ddim.py:22-26 hard-codes "cuda"
    betas = SO.linear_sd_betas()

    class _LDM(_SchedModel):
        def apply_model(self, x, t, c, **kw):
            return analytic_model(x, t, c)
    model = _LDM(betas)
    g = torch.Generator('cpu').manual_seed(123)
    x = torch.randn((2, 4, 5, 6, 7), generator=g)
    c = torch.full((2, 77, 8), 0.25)
    uc = torch.full((2, 77, 8), -0.5)
    out = {'x_seed': 123, 'shape': tuple(x.shape), 'c_val': 0.25, 'uc_val': -0.5}
    for S, scale, eta in ((50, 15.0, 0.0), (20, 7.5, 0.0), (10, 3.0, 0.5)):
        smp = DDIMSampler(model)
        smp.noise_gen.manual_seed(11)
        r, _ = smp.sample(S=S, batch_size=2, shape=tuple(x.shape[1:]), conditioning=c, x_T=x, verbose=False,
                          unconditional_guidance_scale=scale, unconditional_conditioning=uc, eta=eta)
        o = VC.vc_ddim_sample(model, betas, x, S, c, uc, scale, eta=eta, noise_gen=torch.Generator('cpu').manual_seed(11))
        print(f'[vc_ddim] S={S} g={scale} eta={eta}: oracle-vs-reference max|d| = {(r - o).abs().max().item():.3e}')
        assert torch.allclose(r, o, rtol=0, atol=1e-6)
        out[f'S{S}_g{scale}_eta{eta}'] = r
    torch.save(out, os.path.join(GOLD, 'vc_ddim.pt'))


def gold_vae_encode(m):
    """AutoencoderKL.encode(...).mean (t2v_model.py:1640-1644; what compute_latents keeps, t2v_pipeline.py:181-183)."""
    cfg = VO.VAEConfig()
    ddconfig = {'double_z': True, 'z_channels': 4, 'resolution': 256, 'in_channels': 3, 'out_ch': 3, 'ch': 128,
                'ch_mult': [1, 2, 4, 4], 'num_res_blocks': 2, 'attn_resolutions': [], 'dropout': 0.0}
    torch.manual_seed(0)
    ae = m.AutoencoderKL(ddconfig, 4, None).eval()
    specs = VO.encoder_param_specs(cfg)
    sd = ae.state_dict()
    enc_keys = {k for k in sd if k.startswith('encoder.') or k.startswith('quant_conv.')}
    assert enc_keys == set(specs), enc_keys ^ set(specs)
    for k in specs:
        assert tuple(sd[k].shape) == specs[k], k
    W = UO.make_weights(specs, seed=5)
    sd.update(W)
    ae.load_state_dict(sd, strict=True)
    x = torch.rand((2, 3, 64, 96), generator=torch.Generator('cpu').manual_seed(6)) * 2 - 1
    with torch.no_grad():
        post = ae.encode(x)
    mom = VO.vae_encode_moments(W, cfg, x)
    err = (mom[:, :4] - post.mean).abs().max().item()
    print(f'[vae_encode] oracle-vs-reference max|d| = {err:.3e} (mean absmax {post.mean.abs().max().item():.3f})')
    assert err <= 1e-5 * max(1.0, post.mean.abs().max().item())
    assert torch.allclose(torch.clamp(mom[:, 4:], -30.0, 20.0), post.logvar, atol=1e-5)
    torch.save({'wseed': 5, 'x_seed': 6, 'x_shape': (2, 3, 64, 96), 'mean': post.mean, 'logvar': post.logvar},
               os.path.join(GOLD, 'vae_encode.pt'))


def gold_vid2vid_encode():
    """vid2vid entry noise of the three samplers (samplers_common.py:123-145): DDIMSampler.stochastic_encode
    (ddim/sampler.py:270-283), UniPCSampler.unipc_encode (uni_pc/sampler.py:20-29), GaussianDiffusion.add_noise
    (gaussian_sampler.py:87-91) -- reference outputs for tests/test_modules_cpu.py."""
    ref_shim.load_samplers()
    from samplers.ddim.gaussian_sampler import GaussianDiffusion
    from samplers.ddim.sampler import DDIMSampler
    from samplers.uni_pc.sampler import UniPCSampler
    import samplers.uni_pc.sampler as ups
    ups.UniPCSampler.register_buffer = lambda self, name, attr: setattr(self, name, attr)
    betas = SO.linear_sd_betas()
    model = _SchedModel(betas)
    g = torch.Generator().manual_seed(3)
    lat = torch.randn(1, 4, 5, 6, 7, generator=g)
    noise = torch.randn(1, 4, 5, 6, 7, generator=g)
    out = {'lat_noise_seed': 3, 'shape': (1, 4, 5, 6, 7)}
    for strength, steps in ((0.6, 20), (0.25, 30), (1.0, 10)):
        n = int(strength * steps)
        rd = DDIMSampler(model, device=torch.device('cpu'))
        rd.make_schedule(steps)
        r1 = rd.stochastic_encode(lat, torch.tensor([n]), noise=noise) if n < steps else None
        r2 = UniPCSampler(model).unipc_encode(lat, torch.device('cpu'), strength, steps, noise=noise)
        rg = GaussianDiffusion(model, betas)
        r3 = rg.add_noise(lat, noise, rg.get_time_steps(n, 1)[0])
        out[f's{strength}_n{steps}'] = {'ddim': r1, 'unipc': r2, 'gauss': r3}
    torch.save(out, os.path.join(GOLD, 'vid2vid_encode.pt'))


def gold_module_tree(m):
    """State-dict shapes of the reference's UNetSD (dim 64) and AutoencoderKL, and the class of each Linear / Conv
    module of the UNet: the layout the nn.Module mirrors must expose (tests/test_modules_cpu.py)."""
    ddconfig = {'double_z': True, 'z_channels': 4, 'resolution': 256, 'in_channels': 3, 'out_ch': 3, 'ch': 128,
                'ch_mult': [1, 2, 4, 4], 'num_res_blocks': 2, 'attn_resolutions': [], 'dropout': 0.0}
    torch.manual_seed(0)
    net = build_ref_unet(m, UO.UNetConfig(dim=64))
    kinds = ('Linear', 'Conv1d', 'Conv2d', 'Conv3d')
    ae = m.AutoencoderKL(ddconfig, 4, None)
    out = {'unet_dim64': {'state_dict': {k: tuple(v.shape) for k, v in net.state_dict().items()},
                          'modules': {n: type(x).__name__ for n, x in net.named_modules() if type(x).__name__ in kinds}},
           'vae': {'state_dict': {k: tuple(v.shape) for k, v in ae.state_dict().items()}}}
    torch.save(out, os.path.join(GOLD, 'module_tree.pt'))
    print(f'[module_tree] unet {len(out["unet_dim64"]["state_dict"])} tensors, vae {len(out["vae"]["state_dict"])} tensors')


def gold_unet_tiny_b2(m):
    """The reference UNetSD (dim 64) at B = 2 with two different timesteps, seeded weights and inputs."""
    cfg = UO.UNetConfig(dim=64)
    torch.manual_seed(0)
    net = build_ref_unet(m, cfg)
    W = UO.make_weights(UO.param_specs(cfg), seed=5)
    net.load_state_dict(W, strict=True)
    g = torch.Generator().manual_seed(9)
    x = torch.randn(2, 4, 3, 8, 8, generator=g)
    y = torch.randn(2, 77, 1024, generator=g)
    t = torch.tensor([500, 20])
    with torch.no_grad():
        ref = net(x, t, y)
    err = (UO.unet_forward(W, cfg, x, t, y) - ref).abs().max().item()
    print(f'[unet_tiny_b2] oracle-vs-reference max|d| = {err:.3e}')
    torch.save({'wseed': 5, 'xy_seed': 9, 'x_shape': tuple(x.shape), 'y_shape': tuple(y.shape), 't': t, 'out': ref},
               os.path.join(GOLD, 'unet_tiny_b2.pt'))


KEY_FRAME_CASES = [
    (8, 4, '0:(t/max_i_f), "max_i_f":(1)'), (24, 8, '0:(t/max_i_f), "max_i_f":(1)'), (6, 4, '0:(0.25), 3:(1.0)'),
    (10, 3, '0:(0), 4:(0.5), "max_f":(1)'), (12, 6, '0:(sin(t/max_f)), 9:(0.2)'),
    (8, 4, '0:(t/max_i_f), "max_i_f":(1*1)'), (16, 5, '0:(0.1+t/max_f), 11:(t*t/(max_f*max_f))')]


def gold_key_frames():
    """Per-frame inpainting weights of the reference's T2VAnimKeys (t2v_helpers/key_frames.py) for KEY_FRAME_CASES.
    A spec the reference cannot evaluate with the installed pandas is stored with weights None: numeric keys make it
    store a string into a float64 Series (key_frames.py:38), which pandas >= 3 rejects with a TypeError."""
    import json
    import pandas
    from types import SimpleNamespace as NS
    kf = ref_shim.load_key_frames()
    cases = []
    for frames, i_frames, spec in KEY_FRAME_CASES:
        try:
            w = [float(v) for v in kf.T2VAnimKeys(NS(max_frames=frames, inpainting_weights=spec), 7, i_frames)
                 .inpainting_weights_series]
        except TypeError:
            w = None
        cases.append({'frames': frames, 'i_frames': i_frames, 'spec': spec, 'weights': w})
    with open(os.path.join(GOLD, 'key_frames.json'), 'w') as f:
        json.dump({'pandas': pandas.__version__, 'cases': cases}, f, indent=1)
    print(f'[key_frames] {sum(c["weights"] is not None for c in cases)} of {len(cases)} specs evaluated by the reference')


def main(only=None):
    os.makedirs(GOLD, exist_ok=True)
    m = ref_shim.load_modelscope()
    want = lambda n: only is None or n in only      # noqa: E731
    if want('samplers'):
        gold_samplers()
    if want('vae_decode'):
        gold_vae(m)
    if want('vae_encode'):
        gold_vae_encode(m)
    if want('vid2vid_encode'):
        gold_vid2vid_encode()
    if want('module_tree'):
        gold_module_tree(m)
    if want('unet_tiny_b2'):
        gold_unet_tiny_b2(m)
    if want('key_frames'):
        gold_key_frames()
    tiny = UO.UNetConfig(dim=64)
    keep = ['input_blocks.0.0', 'input_blocks.0.1', 'input_blocks.1.0', 'input_blocks.1.1', 'input_blocks.1.2',
            'input_blocks.3', 'input_blocks.4.0', 'input_blocks.11.0', 'middle_block.1', 'middle_block.3',
            'output_blocks.0.0', 'output_blocks.2.1', 'output_blocks.5.3', 'output_blocks.11.2']
    if want('unet_tiny'):
        gold_unet(m, 'unet_tiny', tiny, F=3, h=16, w=8, wseed=1, keep_taps=keep)
    # 125 frames through the temporal conv / temporal attention / 5-D GroupNorm path on the narrow net (config 4's frame count)
    if want('unet_f125'):
        gold_unet_forward_only(m, 'unet_f125', tiny, F=125, h=8, w=8, wseed=1, B=2)
    full = os.environ.get('T2V_GOLD_FULL', '1') == '1'
    if full and want('unet_cfg1'):
        gold_unet(m, 'unet_cfg1', UO.UNetConfig(), F=4, h=16, w=16, wseed=0, keep_taps=[])
    if full and want('unet_cfg2'):       # the shape every bench number is quoted on: 24 frames x 256^2
        gold_unet_step(m, 'unet_cfg2', UO.UNetConfig(), F=24, h=32, w=32, wseed=0)
    if full and want('unet_cfg3_slice'):  # config 3's spatial sequence length S = 72 * 128 = 9216, 2 frames
        gold_unet_forward_only(m, 'unet_cfg3_slice', UO.UNetConfig(), F=2, h=72, w=128, wseed=0)
    if want('vc_ddim'):
        gold_vc_ddim()
    if want('vc_unet_tiny'):
        gold_vc_unet('vc_unet_tiny', VC.VCConfig(model_channels=64, context_dim=48, temporal_length=4), B=2, T=4, h=8, w=8, L=7, wseed=3)
    if full and want('vc_unet_full'):
        gold_vc_unet('vc_unet_full', VC.VCConfig(), B=1, T=16, h=16, w=16, L=77, wseed=0)
    if full and want('vc_unet_cfg5'):     # config 5's per-GPU shape: 16 frames x 256^2
        gold_vc_unet('vc_unet_cfg5', VC.VCConfig(), B=1, T=16, h=32, w=32, L=77, wseed=0, half_out=True)


if __name__ == '__main__':
    main(set(sys.argv[1:]) or None)
