#!/usr/bin/env python
"""bench.py -- images/sec of the imagen sampling hot path on B200 (BASELINE.json metric).

A "step" is one pass of the hot path over one batch: Imagen.sample() of `bs` images through the full
T-step DDPM loop (classifier-free guidance => 2*bs U-Net rows per denoising step).  Workload at every N:
BASELINE.json configs[1]: base Unet(dim=128) 64x64, bs=16 per GPU, 1000 DDPM steps, cond_scale=3.0,
synthetic text_embeds (bs,256,768), random-init weights (final_conv re-randomised: the reference zero-inits it).

    python bench.py --gpus 1 --steps 3 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference algorithm (oracle port) on the host cores
    python bench.py --dump-outputs DIR ...    # also write the last timed step's images as DIR/images.npy (float32)

Prints ONE JSON line (rank 0).  Timing: CUDA events on the launching stream, barrier + synchronize on both sides,
max over ranks.  `value` = inputs resident in HBM; `e2e` = same call with pinned-host text_embeds copied in and the
images copied back inside the timed region.  `roofline` = the dominant kernel (multi-query flash attention at the
64x64 level, 59% of the algorithmic FLOPs) timed alone with CUDA events at the workload's exact shape.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# algorithmic work (SURVEY.md section 8d / BASELINE.md section 3; FlopCounterMode over the reference forward)
GFLOP_PER_FORWARD_DIM128 = 131.90
ATTN_L0_GFLOP_PER_SAMPLE = 2 * 2 * (8 * 4096) * (4096 + 39) * 64 / 1e9          # QK^T + PV of one 64x64 Attention block (:565,:588)


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d['hbm_gbs'], tensor_burst=d['bf16_tflops'], tensor_sustained=d['bf16_tflops_sustained'], src='measured')
    return dict(hbm=6650.0, tensor_burst=1590.0, tensor_sustained=1400.0, src='fallback')


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = 'index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,' \
        'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, f'/tmp/b200_clocks_{os.getpid()}.csv'

    def __enter__(self):
        try:
            self.f = open(self.path, 'w')
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '200', '-i', str(self.index)],
                                         stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
            self.f.close()

    def summary(self):
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                p = [s.strip() for s in line.split(',')]
                if len(p) < 9:
                    continue
                sm.append(float(p[1])); mx.append(float(p[2]))
                for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), p[5:9]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
        except Exception:
            pass
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['unavailable'])
        return dict(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))


def build_model(dim, timesteps, device):
    import imagen_pytorch_b200 as b2
    torch.manual_seed(0)
    unet = b2.Unet(dim=dim)
    with torch.no_grad():                                   # the reference zero-inits final_conv (imagen_pytorch.py:1438)
        unet.final_conv.weight.normal_(0, 0.02)
        unet.final_conv.bias.normal_(0, 0.02)
    return b2.Imagen(unet, image_sizes=64, timesteps=timesteps).to(device)


def build_workload(args, device):
    """(sampler, sample kwargs, images per call, description) of BASELINE.json configs[args.config]."""
    import imagen_pytorch_b200 as b2

    def rand_final(u):
        with torch.no_grad():
            u.final_conv.weight.normal_(0, 0.02)
            u.final_conv.bias.normal_(0, 0.02)
        return u

    torch.manual_seed(0)
    c = args.config
    if c == 1:
        return build_model(args.dim, args.timesteps, device), dict(cond_scale=3.), args.bs, None
    if c == 2:       # configs[2]: ElucidatedImagen base Unet dim=128 64x64, 64 sampler steps, bs=64 (CUDA-graph t-loop: 63 Heun steps + last)
        el = b2.ElucidatedImagen(rand_final(b2.Unet(dim=args.dim)), image_sizes=64, num_sample_steps=args.sample_steps).to(device)
        return el, dict(cond_scale=args.cond_scale), args.bs, \
            f'BASELINE.json configs[2]: ElucidatedImagen base Unet dim={args.dim} 64x64, {args.sample_steps} sampler steps ({2 * args.sample_steps - 1} U-Net evaluations), ' \
            f'bs={args.bs}/GPU, cond_scale={args.cond_scale}'
    if c == 3:       # configs[3]: two-stage cascade 64 -> 256, SR-Unet dim=128 (SRUnet256), bs=8, 100 DDPM steps each
        im = b2.Imagen((rand_final(b2.Unet(dim=args.dim)), rand_final(b2.SRUnet256(lowres_cond=True))), image_sizes=(64, 256),
                       timesteps=args.timesteps).to(device)
        return im, dict(cond_scale=args.cond_scale), args.bs, \
            f'BASELINE.json configs[3]: cascade base Unet dim={args.dim} @64 -> SRUnet256 (dim 128, lowres_cond) @256, bs={args.bs}/GPU, ' \
            f'{args.timesteps} DDPM steps each, cond_scale={args.cond_scale}'
    if c == 4:       # configs[4]: the per-GPU shard of base Unet dim=192 64x64, 1000 steps, global bs 512 over 8 GPUs
        return build_model(args.dim, args.timesteps, device), dict(cond_scale=3.), args.bs, \
            f'BASELINE.json configs[4] per-GPU shard: base Unet dim={args.dim} 64x64, bs={args.bs}/GPU (global 512 over 8 GPUs), {args.timesteps} DDPM steps, cond_scale=3.0'
    raise ValueError(f'unknown --config {c}')


def gpu_eager_step_time(dim, bs, device, steps):
    """The reference's eager fp32 PyTorch ops (oracle port, torch CUDA kernels: cuDNN TF32 convs, cuBLAS, materialised N x M attention)
    on THIS GPU in THIS process: `steps` denoising steps at the full batch -> seconds per denoising step (the denominator of the
    north star's ">= 15x PyTorch-eager on 1xB200")."""
    cpu_reference_step(dim, bs, device=str(device), steps=2)            # warm-up (cuDNN autotune, allocator)
    return cpu_reference_step(dim, bs, device=str(device), steps=steps)


def time_attention_kernel(bs_rows, device, iters=10, max_logit=8 * 1.4426950408889634 * 1.02):
    """The dominant kernel alone, at the workload's shape: one 64x64 multi-query self-attention block, R = 2*bs rows."""
    from imagen_pytorch_b200 import _lib
    import torch.nn.functional as F
    n, heads, nk = 4096, 8, 4096 + 39
    q = (F.normalize(torch.randn(bs_rows, heads * n, 64, device=device), dim=-1) * 8 * 1.4426950408889634).to(torch.bfloat16)
    k = F.normalize(torch.randn(bs_rows, nk, 64, device=device), dim=-1).to(torch.bfloat16)
    v = torch.randn(bs_rows, nk, 64, device=device).to(torch.bfloat16)
    o = torch.empty_like(q)
    st = torch.cuda.current_stream(device)
    args = (q.data_ptr(), o.data_ptr(), heads * n * 64, 0, 64, heads * n, k.data_ptr(), v.data_ptr(), nk * 64, 0, 64, nk, bs_rows, 1, max_logit, st.cuda_stream)
    for _ in range(3):
        _lib.call('b200_attention', *args)
    torch.cuda.synchronize(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(iters):                                  # q+o = 268 MB per launch > 126 MB L2: no explicit flush needed
        _lib.call('b200_attention', *args)
    e1.record(st)
    torch.cuda.synchronize(device)
    return e0.elapsed_time(e1) / iters


def time_conv_kernel(R, device, iters=20):
    """The heaviest conv shape of the workload alone: 64x64 level Block.project, 3x3, 128 -> 128 channels, R rows (NHWC bf16)."""
    from imagen_pytorch_b200 import ops, _lib
    x = torch.randn(R, 64, 64, 128, device=device).to(torch.bfloat16)
    Wt = torch.randn(128, 128, 3, 3, device=device) / 34.0
    segs, mats = ops.conv_segments(Wt, [128])
    wp = ops.pack_weight(mats, 128, device)
    out = torch.empty(R * 4096, 128, dtype=torch.bfloat16, device=device)
    call = ops.GemmCall([(x.data_ptr(), 128, 128)], segs, (R, 64, 64), wp, 128, out.data_ptr(), bias=ops.padded_bias(torch.zeros(128, device=device), 128, device), ldc=128)
    st = torch.cuda.current_stream(device)
    for _ in range(3):
        call(st.cuda_stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)      # > 126 MB L2: flushed between launches
    times = []
    for _ in range(iters):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        call(st.cuda_stream)
        e1.record(st)
        torch.cuda.synchronize(device)
        times.append(e0.elapsed_time(e1))
    return statistics.median(times), 2.0 * R * 4096 * 128 * 1152 / 1e9


def usable_cores():
    """Host cores this process may actually use: affinity mask capped by the cgroup CPU quota (a 128-thread pool on an
    8-CPU quota thrashes: round 1 measured 50 s per step that way)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()
        if quota != 'max':
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


def cpu_reference_step(dim, bs, threads=None, device='cpu', steps=1):
    """`steps` DDPM denoising steps (cond + null U-Net pass, CFG combine, thresholded posterior update) of the reference
    algorithm through the oracle port: on the host cores (device='cpu', the baseline), or -- informational only, flag
    --eager-gpu -- the same eager fp32 PyTorch ops on the GPU (the "PyTorch-eager on B200" denominator of the north star).
    Returns seconds per step."""
    from oracle import unet_ref, sampler_ref
    import imagen_pytorch_b200 as b2
    if threads:
        torch.set_num_threads(threads)
    torch.manual_seed(0)
    u = b2.Unet(dim=dim)
    sd = {k: v.detach().clone().to(device) for k, v in u.state_dict().items()}
    sd['final_conv.weight'].normal_(0, 0.02)
    cfg = unet_ref.unet_config(dim=dim)
    te = torch.randn(bs, 256, 768, device=device)
    fn = lambda x, t, cond_scale, lowres_noise_times=None, **k: unet_ref.unet_forward_with_cond_scale(sd, cfg, x, t, cond_scale=cond_scale, **k)
    randn = (lambda s: torch.randn(tuple(s), device=device))
    kw = dict(text_embeds=te, text_mask=torch.ones(bs, 256, dtype=torch.bool, device=device))
    if device != 'cpu':
        torch.cuda.synchronize()
    t0 = time.perf_counter()
    with torch.no_grad():
        sampler_ref.ddpm_p_sample_loop(fn, (bs, 3, 64, 64), timesteps=steps, cond_scale=3., unet_kwargs=kw, randn=randn)
    if device != 'cpu':
        torch.cuda.synchronize()
    return (time.perf_counter() - t0) / steps


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    if args.eager_gpu:
        # informational: the reference's algorithm as eager fp32 PyTorch ops on this GPU (cuDNN TF32 convs, cuBLAS fp32 bmm,
        # materialised N x M attention scores), full batch, a few denoising steps extrapolated to the schedule length
        cpu_reference_step(args.dim, args.bs, device='cuda', steps=2)
        dt = cpu_reference_step(args.dim, args.bs, device='cuda', steps=max(2, args.steps))
        print(json.dumps({'impl': 'reference-eager-gpu', 'metric': 'images/sec', 'value': args.bs / (dt * args.timesteps), 'unit': 'images/s',
                          'ms_per_denoising_step': dt * 1e3, 'dtype': 'f32 (TF32 conv)', 'config': workload_config(args),
                          'note': 'oracle port executed with torch CUDA ops; not the product path, not the CPU baseline'}))
        return
    cores = usable_cores()
    torch.set_num_threads(cores)
    bs = 1
    for _ in range(args.warmup):
        cpu_reference_step(args.dim, bs)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_reference_step(args.dim, bs)
    dt = (time.perf_counter() - t0) / args.steps
    value = bs / (dt * args.timesteps)                      # one denoising step timed; a batch needs `timesteps` of them
    sample = f'1 of {args.timesteps} DDPM denoising steps (cond+null U-Net pass, cond_scale 3.0) at bs={bs}, extrapolated x{args.timesteps}'
    print(json.dumps({
        'impl': 'reference', 'metric': 'images/sec', 'value': value, 'unit': 'images/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': dt * 1e3 * args.timesteps / bs * args.bs, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic', 'config': workload_config(args),
        'cpu_baseline': {'value': value, 'unit': 'images/s', 'cores': torch.get_num_threads(), 'kind': 'port', 'sample': sample},
        'e2e': {'value': value, 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }))


DUMP_MAX_ELEMENTS = (64 << 20) // 4                          # 64 MB of float32


def dump_images(out_dir, images):
    """Writes what sample() returned as out_dir/images.npy (float32), so that two builds run with the same arguments can be
    compared output for output. Above 64 MB it keeps a fixed, seeded sample of the flattened elements instead: the same
    positions, in ascending order, for every build."""
    import numpy as np
    a = images.detach().float().cpu()
    if a.numel() > DUMP_MAX_ELEMENTS:
        keep = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ELEMENTS].sort().values
        a = a.reshape(-1)[keep]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, 'images.npy'), a.numpy())


def workload_config(args, desc=None):
    if desc is not None:
        return {'workload': desc + f', random text_embeds ({args.bs},256,768)', 'global_batch': args.bs * args.gpus,
                'parallelism': f'dp{args.gpus} (independent sample shards, one all-gather of finished images)',
                'l2': 'no explicit flush: the per-step activation working set (GBs) exceeds the 126 MB L2'}
    return {'workload': f'BASELINE.json configs[1]: base Unet dim={args.dim} 64x64, bs={args.bs}/GPU, {args.timesteps} DDPM steps, cond_scale=3.0 '
                        f'(classifier-free guidance: {2 * args.bs} U-Net rows/step), random text_embeds ({args.bs},256,768)',
            'global_batch': args.bs * args.gpus, 'parallelism': f'dp{args.gpus} (independent sample shards, one all-gather of finished images)',
            'l2': 'no explicit flush: per-step activation working set (GBs) and the 268 MB q/o of the timed attention kernel exceed the 126 MB L2'}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--config', type=int, default=1, choices=[1, 2, 3, 4], help='index into BASELINE.json configs (1 = the headline metric)')
    ap.add_argument('--bs', type=int, default=None)
    ap.add_argument('--dim', type=int, default=None)
    ap.add_argument('--timesteps', type=int, default=None)
    ap.add_argument('--sample-steps', type=int, default=64, help='config 2: ElucidatedImagen num_sample_steps')
    ap.add_argument('--cond-scale', type=float, default=3.0, help='configs 2 and 3')
    ap.add_argument('--eager-steps', type=int, default=20, help='denoising steps of the in-process eager-PyTorch-on-GPU baseline (0 = skip)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--eager-gpu', action='store_true', help='with --impl reference: run the oracle port with torch CUDA ops (informational)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the images of the last timed step to DIR/images.npy (float32)')
    args = ap.parse_args()
    defaults = {1: (16, 128, 1000), 2: (64, 128, None), 3: (8, 128, 100), 4: (64, 192, 1000)}[args.config]
    args.bs = args.bs if args.bs is not None else defaults[0]
    args.dim = args.dim if args.dim is not None else defaults[1]
    args.timesteps = args.timesteps if args.timesteps is not None else (defaults[2] or 1000)
    if args.impl == 'reference':
        return run_reference(args)

    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    assert torch.cuda.is_available(), 'bench.py --impl b200 needs a GPU (no CPU fallback)'
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=device)
    assert args.warmup >= 3, 'timing hygiene: at least 3 warm-up steps'

    from imagen_pytorch_b200.dist import all_gather_images
    imagen, skw, bs_call, desc = build_workload(args, device)
    out_px = imagen.image_sizes[-1]
    torch.manual_seed(1234 + rank)
    te_host = torch.randn(args.bs, 256, 768).pin_memory()
    te_dev = te_host.to(device)
    out_host = torch.empty(args.bs, 3, out_px, out_px).pin_memory()

    own_events = []                                             # (before, after) this rank's own sampling work, all-gather excluded
    last = {}

    def step_resident():
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ea.record()
        img = imagen.sample(text_embeds=te_dev, use_tqdm=False, **skw)
        eb.record()
        own_events.append((ea, eb))
        if world > 1:
            img = all_gather_images(img, [args.bs] * world)
        last['images'] = img
        return img

    def step_e2e():
        te = te_host.to(device, non_blocking=True)          # H2D of this step's inputs from pinned memory
        img = imagen.sample(text_embeds=te, use_tqdm=False, **skw)
        if world > 1:
            img = all_gather_images(img, [args.bs] * world)
        out_host.copy_(img[rank * args.bs:(rank + 1) * args.bs] if world > 1 else img, non_blocking=True)   # D2H of the result
        torch.cuda.current_stream(device).synchronize()
        return img

    def timed(fn, n):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize(device)
        ms = torch.tensor([e0.elapsed_time(e1)], device=device)
        per_rank = [ms.item()]
        if world > 1:
            allms = torch.empty(world, device=device)
            dist.all_gather_into_tensor(allms, ms)              # every rank's own device time: a slow GPU shows up by index
            per_rank = allms.tolist()
            dist.barrier()
        return max(per_rank), per_rank                         # the job's time is the slowest rank's

    for _ in range(args.warmup):
        step_resident()
    own_events.clear()
    with ClockSampler(local) as clk:
        ms, ms_ranks = timed(step_resident, args.steps)
    clocks = clk.summary()
    if args.dump_outputs and rank == 0:                         # before the e2e steps sample again
        dump_images(args.dump_outputs, last['images'])
    own_ms = [sum(a.elapsed_time(b) for a, b in own_events) / args.steps]   # this rank's shard alone: a slow GPU shows up by index
    if world > 1:
        own_all = torch.empty(world, device=device)
        dist.all_gather_into_tensor(own_all, torch.tensor(own_ms, device=device))
        own_ms = own_all.tolist()
    launches = imagen.last_launch_count * args.steps
    step_e2e()
    ms_e2e, ms_e2e_ranks = timed(step_e2e, args.steps)
    rank_clocks = [clocks]
    if world > 1:                                               # per-rank clocks under load next to the per-rank times
        rank_clocks = [None] * world
        dist.all_gather_object(rank_clocks, clocks)

    images = args.bs * world * args.steps
    value = images / (ms / 1e3)
    e2e_value = images / (ms_e2e / 1e3)
    pk = peaks()
    line = {
        'metric': 'images/sec', 'value': value, 'unit': 'images/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16',
        'data': 'synthetic', 'config': workload_config(args, desc), 'clocks': clocks, 'gpu_launches': launches,
        'e2e': {'value': e2e_value, 'unit': 'images/s', 'h2d_bytes_per_step': te_host.numel() * 4, 'd2h_bytes_per_step': out_host.numel() * 4},
        'per_rank': {'ms_per_step': [m / args.steps for m in ms_ranks], 'ms_per_step_min': min(ms_ranks) / args.steps,
                     'ms_per_step_median': statistics.median(ms_ranks) / args.steps, 'ms_per_step_max': max(ms_ranks) / args.steps,
                     'own_sampling_ms_per_step': own_ms,
                     'e2e_ms_per_step': [m / args.steps for m in ms_e2e_ranks],
                     'sm_mhz': [c.get('sm_mhz') for c in rank_clocks], 'reasons': [c.get('reasons') for c in rank_clocks]},
    }
    if rank == 0 and args.config != 1:
        print(json.dumps(line))
    if rank == 0 and args.config == 1:
        R = 2 * args.bs
        att_ms = time_attention_kernel(R, device)
        att_tflops = ATTN_L0_GFLOP_PER_SAMPLE * R / 1e3 / (att_ms / 1e3)
        # MUFU floor of head-dim-64 attention: one exp2 per score, 16 exp2/clk/SM measured (profiles/r01_mufu_ex2_microbench.txt)
        n_exp = R * 8 * 4096 * ((4096 + 39 + 127) // 128 * 128)
        mufu_ms = n_exp / (148 * 16 * 1.965e9) * 1e3
        line['roofline'] = {'kernel': 'flash_attn_pt_kernel<4,2,0,1105> (tcgen05 multi-query self-attention, P in tensor memory, scores preloaded, S MMAs on a third issuer thread; 64x64 level: 8*4096 query rows x 4135 keys x d64 per sample)',
                            'bound': 'tensor', 'achieved': att_tflops, 'peak': pk['tensor_burst'], 'unit': 'TFLOP/s', 'frac': att_tflops / pk['tensor_burst'],
                            'traffic': 261.9e6, 'traffic_source': 'ncu --set full dram__bytes_read.sum + dram__bytes_write.sum of one launch (profiles/r02_ncu_flash_attn_pt_summary.txt); algorithmic q+o+k+v = 285 MB',
                            'ms_per_launch': att_ms, 'algorithmic_gflop_per_launch': ATTN_L0_GFLOP_PER_SAMPLE * R,
                            'peak_source': f"{pk['src']} burst bf16 (kernel timed alone)",
                            'mufu_floor_ms': mufu_ms, 'frac_of_mufu_floor': mufu_ms / att_ms}
        conv_ms, conv_gflop = time_conv_kernel(R, device)
        line['roofline_conv'] = {'kernel': 'conv_gemm_tc_kernel<128,6,1,8,0> (tcgen05 implicit-GEMM conv3x3 128->128 @64x64, 128 x 128 tiles, MMAs issued under elect.sync)', 'bound': 'tensor',
                                 'achieved': conv_gflop / conv_ms, 'peak': pk['tensor_burst'], 'unit': 'TFLOP/s', 'frac': conv_gflop / conv_ms / pk['tensor_burst'],
                                 'traffic': 34.0e6, 'ms_per_launch': conv_ms, 'algorithmic_gflop_per_launch': conv_gflop,
                                 'note': 'L2 flushed between launches; dram traffic from ncu --set full = 33.9 MB read + 1.4 MB written (profiles/r02_ncu_conv_gemm_summary.txt: input 33.5 MB read once, the 33.5 MB output stays in L2)'}
        step_tflop = GFLOP_PER_FORWARD_DIM128 * 2 * args.bs * args.timesteps / 1e3 if args.dim == 128 else None
        if step_tflop:
            ach = step_tflop / (ms / args.steps / 1e3)
            line['whole_step'] = {'algorithmic_tflop_per_step': step_tflop, 'achieved_tflops': ach, 'frac_of_sustained_bf16': ach / pk['tensor_sustained']}
        if args.eager_steps > 0:
            # the north star's ">= 15x the reference PyTorch-eager images/sec on 1xB200": same GPU, same process, same batch
            with ClockSampler(local) as eclk:
                dt = gpu_eager_step_time(args.dim, args.bs, device, args.eager_steps)
            eager = args.bs / (dt * args.timesteps)
            line['gpu_eager_baseline'] = {'value': eager, 'unit': 'images/s', 'ms_per_denoising_step': dt * 1e3, 'denoising_steps_timed': args.eager_steps,
                                          'batch': args.bs, 'dtype': 'f32 (TF32 convolutions, cuDNN / cuBLAS / ATen eager kernels)', 'clocks': eclk.summary(),
                                          'speedup_value': value / world / eager, 'speedup_e2e': e2e_value / world / eager,
                                          'what': f'oracle port of the reference forward + DDPM step executed with torch CUDA ops on this GPU: {args.eager_steps} denoising steps '
                                                  f'(cond + null pass, cond_scale 3.0) at bs={args.bs}, extrapolated x{args.timesteps}; informational baseline, not the product path'}
        if not args.no_cpu_baseline:
            cores = usable_cores()
            torch.set_num_threads(cores)
            cpu_reference_step(args.dim, 1)
            t = min(cpu_reference_step(args.dim, 1) for _ in range(2))
            line['cpu_baseline'] = {'value': 1 / (t * args.timesteps), 'unit': 'images/s', 'cores': torch.get_num_threads(), 'kind': 'port',
                                    'sample': f'1 of {args.timesteps} DDPM denoising steps (cond+null pass) at bs=1 through the oracle port, extrapolated x{args.timesteps}'}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
