#!/usr/bin/env python
"""Benchmark of the text2video denoising hot path: denoised frames/s = F / (sampling loop + VAE decode) for
ModelScope 24 frames x 256x256, 50-step DDIM (UI-default scheduler "DDIM_Gaussian", cfg 17), fp16, synthetic weights.

    python bench.py --gpus 1 --steps K --warmup W                      # this repo (B200, libt2v_b200.so)
    torchrun --nproc-per-node N ... bench.py --gpus N ...              # one independent clip per GPU (sample-DP, weak)
    python bench.py --impl reference ...                               # the reference algorithm on the host cores
    python bench.py --impl torch_gpu ...                               # the reference's GPU path (fp16 autocast + SDPA eager torch ops)

A "step" is one whole clip: 50 scheduler steps (each = one batched cond+uncond UNet forward + fused CFG/DDIM update)
followed by the VAE decode of all frames.  `value` has inputs resident in HBM; `e2e` goes through the public
`TextToVideoSynthesis.infer` with host buffers (H2D of conditioning + noise and D2H of the finished uint8 clip inside
the timed region).  One JSON line is printed by rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (no __pycache__ beside the sources)
for p in (ROOT, os.path.join(ROOT, 'sd-webui-text2video_b200')):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch          # noqa: E402

METRIC = 'denoised frames/sec (UNet+VAE) ModelScope 24fx256^2 50-step'


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3, help='timed clips')
    ap.add_argument('--warmup', type=int, default=3, help='untimed warm-up clips (>= 3)')
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference', 'torch_gpu'])
    ap.add_argument('--frames', type=int, default=24)
    ap.add_argument('--height', type=int, default=256)
    ap.add_argument('--width', type=int, default=256)
    ap.add_argument('--denoise-steps', type=int, default=50)
    ap.add_argument('--sampler', default='DDIM_Gaussian')
    ap.add_argument('--cfg-scale', type=float, default=17.0)
    ap.add_argument('--mode', default='sample_dp', choices=['sample_dp', 'frame_shard', 'frame_shard_cfg'],
                    help='N>1: sample_dp = one clip per GPU (weak scaling, the default the driver runs); frame_shard = ONE clip '
                         'split over the N GPUs by frames (strong scaling, BASELINE config 4: --frames 125); frame_shard_cfg = the same '
                         'with the guidance pair split as well: N/2 frame shards x (cond | uncond), one eps exchange per step')
    ap.add_argument('--no-shard-leg', action='store_true', help='skip the secondary strong-scaling measurement (ONE 125-frame clip '
                                                                'frame-sharded over all N GPUs; at N = 1 the same clip on one GPU)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-gpu-baseline', action='store_true', help='skip the torch-eager GPU comparator leg of the N=1 run')
    ap.add_argument('--cpu-frames', type=int, default=0, help='frames of the CPU sample (0 = the metric\'s F)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='after the timed clips, write what the last one returned (the '
                                                          'decoded uint8 frames) to DIR/<name>.npy as float32')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be >= 1')
    return args


DUMP_LIMIT_BYTES = 60 << 20     # all dumped arrays together stay under 64 MB


def dump_outputs(out_dir, arrays):
    """Writes each tensor as out_dir/<name>.npy in float32.  When the arrays together exceed DUMP_LIMIT_BYTES, each is
    replaced by the same share of its flattened elements at indices drawn from a fixed seed (sorted), so two runs with
    the same arguments dump the same positions."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.numel() for a in arrays.values())
    budget = DUMP_LIMIT_BYTES // 4
    for name, a in arrays.items():
        a = a.detach().float().cpu().numpy()
        if total > budget:
            idx = np.sort(np.random.default_rng(0).integers(0, a.size, a.size * budget // total))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + '.npy'), a)


def peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            p = json.load(f)
        return {'tflops_sustained': p['bf16_tflops_sustained'], 'tflops_burst': p['bf16_tflops'], 'hbm_gbs': p['hbm_gbs'],
                'source': 'measured (MEASURED_PEAKS.json)'}
    except Exception:
        return {'tflops_sustained': 1400.0, 'tflops_burst': 1590.0, 'hbm_gbs': 6650.0,
                'source': 'fallback (B200_PROFILING.md)'}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons every 200 ms while the timed region runs."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-i',
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(',')])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace('.', '').isdigit())
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith('active') for r in self.rows)]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': float(self.rows[0][1]), 'samples': len(self.rows),
                'power_w_max': max(float(r[2]) for r in self.rows), 'reasons': reasons}


# --------------------------------------------------------------------------------------------- reference / CPU arm
def cpu_reference_sample(args, nsteps=1, threads=None):
    """The reference ALGORITHM (oracle/: CPU restatement pinned bit-exact against the reference's modules) on the host
    cores, as BASELINE.md section 4.2 prescribes: ONE DDIM_Gaussian step (cond + uncond UNetSD forward + update, fp32 eager)
    at the metric's own shape (F frames x H x W) plus the VAE decode of one frame, extrapolated with
        frames/s = F_s / (denoise_steps * t_step + F_s * t_vae_frame)        (F_s = F unless --cpu-frames shrinks the sample).
    Returns (fps, t_step, t_vae, threads, F_s, per-sample wall seconds)."""
    from oracle import unet_oracle as UO, vae_oracle as VO, samplers_oracle as SO
    # torch's CPU kernels scale poorly past ~16 threads on these tensors (measured in round 1: 128 threads on the GPU box's
    # host were 50x SLOWER than 8 threads), so the baseline uses min(cores, 16) threads and reports that number
    threads = threads or min(os.cpu_count() or 1, 16)
    torch.set_num_threads(threads)
    Fs, h, w = (args.cpu_frames or args.frames), args.height // 8, args.width // 8
    cfg = UO.UNetConfig()
    W = UO.make_weights(UO.param_specs(cfg), seed=0)
    Wv = UO.make_weights(VO.decoder_param_specs(VO.VAEConfig()), seed=3)
    betas = SO.linear_sd_betas()
    g = torch.Generator().manual_seed(123)
    x = torch.randn(1, 4, Fs, h, w, generator=g)
    c = torch.randn(1, 77, 1024, generator=g)
    uc = torch.randn(1, 77, 1024, generator=g)

    class Stop(Exception):
        pass

    def one():
        t0 = time.perf_counter()
        tr = []

        def cb(step):
            raise Stop()
        try:
            SO.ddim_gaussian_sample(lambda a, b, d: UO.unet_forward(W, cfg, a, b, d), betas, x, args.denoise_steps, c, uc,
                                    args.cfg_scale, callback=cb, trace=tr)
        except Stop:
            pass
        t1 = time.perf_counter()
        VO.vae_decode(Wv, VO.VAEConfig(), tr[0][:, :, 0] / 0.18215)
        t2 = time.perf_counter()
        return t1 - t0, t2 - t1
    times = [one() for _ in range(nsteps)]
    t_step = sorted(t[0] for t in times)[len(times) // 2]
    t_vae = sorted(t[1] for t in times)[len(times) // 2]
    fps = Fs / (args.denoise_steps * t_step + Fs * t_vae)
    return fps, t_step, t_vae, threads, Fs, [a + b for a, b in times]


CPU_FORMULA = 'frames/s = F_s / (denoise_steps * t_step + F_s * t_vae_frame)'


def run_reference(args):
    """`--impl reference`: a "step" here is ONE bounded sample of the workload -- one DDIM_Gaussian step at the metric's F
    plus one VAE frame on the host cores (about half a minute) -- so K is capped at 3 timed + 1 warm-up sample to keep the
    run within a few minutes; `steps` / `ms_per_step` report what actually ran, `value` is the extrapolated metric."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    n = max(1, min(args.steps, 3))
    w = 1 if args.warmup > 0 else 0
    t0 = time.perf_counter()
    if w:
        cpu_reference_sample(args, nsteps=1)
    fps, t_step, t_vae, threads, Fs, walls = cpu_reference_sample(args, nsteps=n)
    wall = time.perf_counter() - t0
    sample = (f'{n} x [1 DDIM_Gaussian step (cond + uncond UNetSD forward, fp32 eager) at {Fs} frames x {args.height}x{args.width} '
              f'+ 1 VAE frame], median t_step {t_step:.2f}s t_vae {t_vae:.2f}s, {threads} threads; {CPU_FORMULA}')
    line = {'impl': 'reference', 'metric': METRIC, 'value': fps, 'unit': 'frames/s', 'n_gpus': args.gpus, 'steps': n,
            'warmup': w, 'steps_requested': args.steps, 'warmup_requested': args.warmup,
            'ms_per_step': 1000.0 * sum(walls) / len(walls), 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic (seeded random-init weights, random conditioning)',
            'config': {'workload': f'ModelScope UNetSD {args.frames}f x {args.height}x{args.width}, {args.denoise_steps}-step '
                                   f'{args.sampler}, cfg {args.cfg_scale}, + VAE decode',
                       'step': 'one bounded CPU sample (see cpu_baseline.sample); value is extrapolated to the whole clip',
                       'F_s': Fs, 'threads': threads, 'formula': CPU_FORMULA, 'ms_per_clip_extrapolated': 1000.0 * args.frames / fps},
            'cpu_baseline': {'value': fps, 'unit': 'frames/s', 'cores': threads, 'kind': 'port', 'sample': sample},
            'e2e': {'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'wall_s': wall}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- reference GPU comparator
def torch_gpu_clip_fn(args, dev):
    """The reference's own GPU path, SURVEY.md section 8d / BASELINE.md section 4.1 (the ">= 15x" denominator): the same torch
    ops as the reference module tree (oracle/, pinned against the reference on CPU) with fp16 weights under
    torch.autocast('cuda') (t2v_pipeline.py:271), attention through F.scaled_dot_product_attention (t2v_model.py:566-569, the
    only backend reachable on sm_100), TWO sequential B = 1 forwards per step (gaussian_sampler.py:161-162), the reference
    sampler arithmetic, and the per-frame VAE loop with a .cpu() per frame (t2v_pipeline.py:347-355).  /root/reference does
    not exist on the GPU box, so the module tree itself cannot be timed there; its restatement issues the same library
    kernels (cuDNN / cuBLAS / SDPA / elementwise).  Model movement and torch_gc() calls of the reference are left out (they
    would only slow it down).  Returns fn(seed) -> list of decoded frames on the host."""
    from oracle import unet_oracle as UO, vae_oracle as VO, samplers_oracle as SO
    cfg = UO.UNetConfig()
    W = {k: v.half().to(dev) for k, v in UO.make_weights(UO.param_specs(cfg), seed=0).items()}
    Wv = {k: v.half().to(dev) for k, v in UO.make_weights(VO.decoder_param_specs(VO.VAEConfig()), seed=3).items()}
    betas = SO.linear_sd_betas()
    g = torch.Generator().manual_seed(2)
    c = torch.randn(1, 77, 1024, generator=g).half().to(dev)
    uc = torch.randn(1, 77, 1024, generator=g).half().to(dev)
    F, h, w = args.frames, args.height // 8, args.width // 8
    UO.ATTN_IMPL = 'sdpa'

    def model(x, t, y):
        return UO.unet_forward(W, cfg, x, t.to(dev), y)

    def clip(seed):
        x_T = torch.randn((1, 4, F, h, w), generator=torch.Generator().manual_seed(seed)).to(dev)    # samplers_common.py:118-119
        with torch.no_grad(), torch.autocast('cuda', dtype=torch.float16):
            if args.sampler == 'DDIM':
                x0 = SO.ddim_sample(model, betas, x_T, args.denoise_steps, c, uc, args.cfg_scale)
            else:
                x0 = SO.ddim_gaussian_sample(model, betas, x_T, args.denoise_steps, c, uc, args.cfg_scale)
            frames = []
            for chunk in torch.chunk(x0, chunks=F, dim=2):                       # one frame per decode call + .cpu()
                frames.append(VO.vae_decode(Wv, VO.VAEConfig(), (chunk / 0.18215)[:, :, 0]).cpu())
        return frames
    return clip


def time_torch_gpu(args, dev, clips, warm_clips=1):
    clip = torch_gpu_clip_fn(args, dev)
    for i in range(warm_clips):
        clip(900 + i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(clips):
        clip(123 + i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / clips
    return args.frames / (ms / 1000.0), ms


TORCH_GPU_KIND = ('reference ops restated (oracle/) as eager torch on the same GPU: fp16 autocast + SDPA, two sequential B=1 forwards '
                  'per step, reference sampler arithmetic, per-frame VAE decode + .cpu()')


def run_torch_gpu(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    n = max(1, min(args.steps, 3))
    fps, ms = time_torch_gpu(args, dev, n, warm_clips=1)
    line = {'impl': 'torch_gpu', 'metric': METRIC, 'value': fps, 'unit': 'frames/s', 'n_gpus': 1, 'steps': n, 'warmup': 1,
            'steps_requested': args.steps, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f16 autocast', 'data': 'synthetic (seeded random-init weights, random conditioning)',
            'config': {'workload': f'ModelScope UNetSD {args.frames}f x {args.height}x{args.width}, {args.denoise_steps}-step '
                                   f'{args.sampler}, cfg {args.cfg_scale}, + per-frame VAE decode', 'kind': TORCH_GPU_KIND},
            'e2e': {'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': int(4 * args.frames * (args.height // 8) * (args.width // 8) * 4),
                    'd2h_bytes_per_step': int(args.frames * args.height * args.width * 3 * 4)}}
    print(json.dumps(line), flush=True)


def recorded_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per gemm_tc_kernel launch (bytes), from the committed ncu capture of the
    434 GEMM launches of one forward (profiles/r01_gemm_dram_traffic.json); None when the file is absent.  A number taken
    under ncu cannot be produced inside a timed run, so it is recorded, not live."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'r01_gemm_dram_traffic.json')) as f:
            return float(json.load(f)['dram_bytes_per_launch'])
    except Exception:
        return None


# --------------------------------------------------------------------------------------------- this repo
def run_b200(args):
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    from t2v_b200.pipeline import TextToVideoSynthesis, SCALE_FACTOR
    from t2v_b200.synthetic import randomize_
    from t2v_b200 import samplers

    pipe = TextToVideoSynthesis(None, device=dev)
    randomize_(pipe.sd_model, seed=0)
    randomize_(pipe.autoencoder, seed=3)
    frame_shard = args.mode in ('frame_shard', 'frame_shard_cfg') and world > 1
    if args.mode == 'frame_shard_cfg' and world > 1:
        if world % 2:
            raise SystemExit('frame_shard_cfg needs an even number of GPUs')
        os.environ['T2V_CFG_SPLIT'] = '1'                  # even ranks: conditional branch, odd ranks: unconditional (distributed.py)
        from t2v_b200 import distributed as D0
        D0.cfg_pair()                                       # collective group creation, same order on every rank
        # 2 GPUs: one shard per branch = the plain CFG-pair split (nothing left to shard over frames)
        fs = pipe.enable_frame_shard(D0.cfg_role_group()) if world > 2 else None
        frame_shard = fs is not None
    else:
        fs = pipe.enable_frame_shard() if frame_shard else None
    F, H, Wd = args.frames, args.height, args.width
    h, w = H // 8, Wd // 8
    S = args.denoise_steps
    g = torch.Generator().manual_seed(2)
    c_host = torch.randn(1, 77, 1024, generator=g).half().pin_memory()
    uc_host = torch.randn(1, 77, 1024, generator=g).half().pin_memory()
    c_dev, uc_dev = c_host.to(dev), uc_host.to(dev)
    entry = [s for s in samplers.available_samplers if s.name == args.sampler][0]

    def clip_device(seed):
        """inputs resident in HBM; result (uint8 frames) stays on the device"""
        x_T = torch.randn((1, 4, F, h, w), device=dev, generator=torch.Generator(device=dev).manual_seed(seed))
        smp = entry.init_sampler(pipe.sd_model, betas=pipe.diffusion.betas, device=dev)
        if fs is not None:          # ONE clip over all ranks: this rank's frames through the loop, one latent all-gather, sharded VAE
            fs.begin(F, seed)
            try:
                x_l = fs.local(x_T)
                x0 = smp.sample(S=S, conditioning=c_dev, unconditional_conditioning=uc_dev,
                                unconditional_guidance_scale=args.cfg_scale, x_T=x_l, shape=tuple(x_l.shape), eta=0.0, batch_size=1)
            finally:
                fs.end()
            return fs.decode(fs.gather_latent(x0), 1.0 / SCALE_FACTOR)
        x0 = smp.sample(S=S, conditioning=c_dev, unconditional_conditioning=uc_dev, unconditional_guidance_scale=args.cfg_scale,
                        x_T=x_T, shape=tuple(x_T.shape), eta=0.0, batch_size=1)
        return pipe.autoencoder.decode_video(x0, 1.0 / SCALE_FACTOR, as_uint8=True)

    def clip_e2e(seed):
        """public API with host buffers: H2D of conditioning + CPU-generated noise, D2H of the finished clip"""
        frames, _, _ = pipe.infer(c_host, uc_host, S, F, seed, args.cfg_scale, Wd, H, 0.0, 'GPU (half precision)', dev,
                                  None, 0, 0.0, None, False, args.sampler)
        return frames

    def gather(frames_u8):
        if world > 1 and fs is None:     # the reference's gather_data: one all-gather of the decoded clips (lvdm/utils/dist_utils.py:14-19)
            out = [torch.empty_like(frames_u8) for _ in range(world)]
            dist.all_gather(out, frames_u8)

    def timed(fn, k, base_seed, with_gather):
        """(ms for k clips, what the last clip returned)"""
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(k):
            r = fn(base_seed + i * n_units + unit)
            if with_gather:
                gather(r)
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.barrier()
        return float(ms.item()), r

    from t2v_b200 import distributed as D
    unit, n_units = D.units()       # clip-rendering units: ranks (sample-DP) or rank pairs (T2V_CFG_SPLIT=1, distributed.py)
    if fs is not None:
        unit, n_units = 0, 1        # every rank works on the same clip (same seed)
    W = max(args.warmup, 1)
    for i in range(W):
        clip_device(1000 + i)
    torch.cuda.synchronize()
    clk = ClockSampler(local)
    clk.start()
    ms, last_frames = timed(clip_device, args.steps, 123, True)
    clk.stop_flag = True
    clk.join(timeout=2)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {'frames': last_frames})
    fps = n_units * args.steps * F / (ms / 1000.0)
    clip_e2e(7)                                   # warm the e2e path (pinned staging, plan for B=2 already built)
    ms_e2e, _ = timed(clip_e2e, args.steps, 123, False)
    fps_e2e = n_units * args.steps * F / (ms_e2e / 1000.0)

    prof = None
    unet = pipe.sd_model
    # work / launch counts of the measured mode: taken before the model is switched to frame-shard mode by the secondary leg below
    # sharded: flops() is this rank's share (frame_shard_cfg: B = 1 per rank, half the ranks per branch)
    unet_flops = (unet.flops(1, F, h, w, 77) * world if args.mode == 'frame_shard_cfg' and fs is not None else
                  unet.flops(2, F, h, w, 77) * (world if fs is not None else 1))
    vae_flops = pipe.autoencoder.flops(F, h, w)
    launches_clip = S * (unet.num_launches() + 3) + 120
    n_exchanges = unet.num_exchanges(F) if fs is not None else 0
    if rank == 0:       # per-launch CUDA-event profile of one forward
        prof = (unet.profile(2, F, h, w, 77) if fs is None else
                {'gemm': {'ms': 0.0, 'flop': 0.0, 'launches': 0}, 'total_ms': 0.0})

    # ---- secondary measurement, default mode only: BASELINE config 4, ONE 125-frame 256x256 clip, strong scaling.  N = 1: the clip
    # on one GPU; N > 1: frame-sharded over all N GPUs (activations exchanged inside the UNet kernels over NVLink peer memory, one
    # NCCL all-gather of the final latent, frame-sharded VAE).  1 warm-up clip (plan build + graph capture) + 1 timed clip.
    shard_leg = None
    if args.mode == 'sample_dp' and not args.no_shard_leg and args.frames == 24:
        F4 = 125
        try:
            fs4 = pipe.enable_frame_shard() if world > 1 else None

            def clip125(seed):
                x_T = torch.randn((1, 4, F4, h, w), device=dev, generator=torch.Generator(device=dev).manual_seed(seed))
                smp = entry.init_sampler(pipe.sd_model, betas=pipe.diffusion.betas, device=dev)
                if fs4 is None:
                    x0 = smp.sample(S=S, conditioning=c_dev, unconditional_conditioning=uc_dev, unconditional_guidance_scale=args.cfg_scale,
                                    x_T=x_T, shape=tuple(x_T.shape), eta=0.0, batch_size=1)
                    return pipe.autoencoder.decode_video(x0, 1.0 / SCALE_FACTOR, as_uint8=True)
                fs4.begin(F4, seed)
                try:
                    x_l = fs4.local(x_T)
                    x0 = smp.sample(S=S, conditioning=c_dev, unconditional_conditioning=uc_dev,
                                    unconditional_guidance_scale=args.cfg_scale, x_T=x_l, shape=tuple(x_l.shape), eta=0.0, batch_size=1)
                finally:
                    fs4.end()
                return fs4.decode(fs4.gather_latent(x0), 1.0 / SCALE_FACTOR)
            clip125(2000)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            clip125(2001)
            e1.record()
            torch.cuda.synchronize()
            ms4 = torch.tensor([e0.elapsed_time(e1)], device=dev)
            if world > 1:
                dist.all_reduce(ms4, op=dist.ReduceOp.MAX)
            ms4 = float(ms4.item())
            shard_leg = {'workload': f'ModelScope UNetSD {F4}f x {H}x{Wd}, {S}-step {args.sampler}, ONE clip' +
                                     (f' frame-sharded over {world} GPUs' if world > 1 else ' on one GPU'),
                         'scaling': 'strong', 'n_gpus': world, 'value': F4 / (ms4 / 1000.0), 'unit': 'frames/s', 'ms_per_clip': ms4,
                         'clips_timed': 1, 'exchanges_per_forward': pipe.sd_model.num_exchanges(F4) if world > 1 else 0,
                         'collectives': 'none inside the sampling loop; 1 NCCL all-gather of the latent + 1 of the decoded frames per clip'
                                        if world > 1 else 'none'}
        except Exception as ex:                     # never lose the headline number over the secondary leg
            shard_leg = {'error': str(ex)[:300]}

    if rank == 0:
        pk = peaks()
        gemm = prof['gemm']
        achieved = gemm['flop'] / (gemm['ms'] * 1e-3) / 1e12 if gemm['ms'] > 0 else 0.0
        clip_flops = S * unet_flops + vae_flops
        # per GPU: a clip-rendering unit (one GPU, or a CFG pair) finishes one clip every ms / steps
        whole_clip_tflops = clip_flops / (ms / args.steps * 1e-3) / 1e12 / (world / n_units)
        line = {
            'metric': METRIC, 'value': fps, 'unit': 'frames/s', 'n_gpus': world, 'steps': args.steps, 'warmup': W,
            'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'strong' if fs is not None else 'weak', 'vs_baseline': None,
            'dtype': 'f16 (fp32 accumulate / norms / softmax)', 'data': 'synthetic (seeded random-init weights of the public '
            'ModelScope architecture, random CLIP-like conditioning)',
            'config': {'workload': f'ModelScope UNetSD {F}f x {H}x{Wd}, {S}-step {args.sampler}, cfg {args.cfg_scale}, batched '
                                   f'cond+uncond forward, + AutoencoderKL decode of {F} frames',
                       'parallelism': ((f'CFG split x frame-shard ({world // 2} shards x 2 branches): ' if args.mode == 'frame_shard_cfg' else '') +
                                       f'frame-shard x{world}: ONE clip, {F} frames split over the GPUs; activations exchanged inside the UNet '
                                       f'kernels over NVLink peer memory ({n_exchanges} layout exchanges per forward, no NCCL call per '
                                       'step), one NCCL all-gather of the final latent before a frame-sharded VAE' if fs is not None else
                                       f'sample-DP x{world} (one clip per GPU, one NCCL all-gather of the decoded clips)' if n_units == world else
                                       f'CFG-pair split: {n_units} pair(s) of GPUs, cond / uncond branch per GPU, one eps all-gather per step'),
                       'l2': 'inputs larger than L2: 2.8 GB of fp16 weights are re-read every forward, activations stream through a '
                             'multi-GB arena', 'flop_per_clip': clip_flops},
            'e2e': {'value': fps_e2e, 'unit': 'frames/s',
                    'h2d_bytes_per_step': int(2 * c_host.numel() * 2 + 4 * F * h * w * 4),
                    'd2h_bytes_per_step': int(F * H * Wd * 3)},
            'gpu_launches': int(launches_clip * args.steps),
            'clocks': clk.summary(),
            'roofline': {'bound': 'tensor', 'achieved': achieved, 'peak': pk['tflops_sustained'], 'unit': 'TFLOP/s',
                         'frac': achieved / pk['tflops_sustained'], 'traffic': recorded_traffic(), 'peak_source': pk['source'],
                         'kernel_frac': achieved / pk['tflops_sustained'],
                         'whole_clip_tflops': whole_clip_tflops, 'whole_clip_frac': whole_clip_tflops / pk['tflops_sustained'],
                         'whole_clip_frac_of_burst': whole_clip_tflops / pk['tflops_burst'],
                         'kernel': 'gemm_tc_kernel (tcgen05 implicit GEMM), all launches of one B=2 forward, CUDA events per launch',
                         'gemm_share_of_forward': gemm['ms'] / prof['total_ms'] if prof['total_ms'] else None,
                         'forward_breakdown_ms': {k: round(v['ms'], 3) for k, v in prof.items() if isinstance(v, dict)}},
        }
        if shard_leg is not None:
            line['frame_shard_125f'] = shard_leg
        if world == 1 and not args.no_gpu_baseline:
            # the ">= 15x" denominator of BASELINE.json's north_star: the reference's fp16 PyTorch path on this same GPU
            try:
                gfps, gms = time_torch_gpu(args, dev, clips=1, warm_clips=1)
                line['gpu_eager_baseline'] = {'value': gfps, 'unit': 'frames/s', 'ms_per_clip': gms, 'kind': TORCH_GPU_KIND,
                                              'sample': '1 warm-up clip + 1 timed clip, CUDA events'}
                line['vs_torch_gpu'] = {'e2e_ratio': fps_e2e / gfps, 'device_resident_ratio': fps / gfps}
            except Exception as ex:
                line['gpu_eager_baseline'] = {'value': None, 'error': str(ex)[:300]}
        if world == 1 and not args.no_cpu_baseline:
            try:
                cfps, t_step, t_vae, threads, Fs, _ = cpu_reference_sample(args, nsteps=1)
                line['cpu_baseline'] = {'value': cfps, 'unit': 'frames/s', 'cores': threads, 'kind': 'port', 'F_s': Fs,
                                        'formula': CPU_FORMULA,
                                        'sample': f'1 DDIM_Gaussian step (2 UNetSD forwards, fp32 eager) at {Fs} frames x {H}x{Wd} + 1 VAE '
                                                  f'frame, extrapolated to {S} steps (t_step {t_step:.2f}s, t_vae {t_vae:.2f}s)'}
            except Exception as ex:                 # the baseline is informational; never lose the GPU number over it
                line['cpu_baseline'] = {'value': None, 'error': str(ex)[:200]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == 'reference':
        run_reference(args)
    elif args.impl == 'torch_gpu':
        run_torch_gpu(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
