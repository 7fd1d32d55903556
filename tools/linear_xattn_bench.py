"""Linear cross-attention (Unet(use_linear_cross_attn=True)) on one B200, all in one process so the numbers are comparable:

1. kernel time at the cfg-2 64x64 level (R = 32 rows = bs 16 with CFG, 4096 pixels, 8 x 64 heads, 39 context keys): the per-step context
   kernel, the linear attention kernel, and b200_attention's cosine-sim cross kernel (cross_attn_tc_kernel) at the same shape, alternated,
   CUDA events over many launches.  q + o = 2 x 134 MB per launch > 126 MB L2, so every launch streams from HBM.
2. one denoising step of Unet(dim=128) with and without use_linear_cross_attn=True: Imagen.sample at bs 16, cond_scale 3, 100 DDPM
   steps (captured step graph), ms per step and launches per step.

    python tools/linear_xattn_bench.py [--out profiles/r03_linear_xattn_ab.txt]
The two attention kernels compute different functions; their outputs are compared with the reference only in
tests/test_linear_cross_attention.py."""
import argparse
import subprocess
import sys
import os

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import imagen_pytorch_b200 as b2  # noqa: E402
from imagen_pytorch_b200 import _lib  # noqa: E402

COPY_GBS = 6567.          # measured HBM copy rate of the B200 (MEASURED_PEAKS.json, profiles/README.md)
LOG2E = 1.4426950408889634


def gpu_info():
    try:
        return subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f'nvidia-smi unavailable ({e})'


def kernels(dev, R=32, n=4096, heads=8, nk=39, iters=200, rounds=5):
    inner = heads * 64
    st = torch.cuda.current_stream(dev).cuda_stream
    lib = _lib.load()
    g = torch.Generator(device=dev).manual_seed(0)
    q = torch.randn(R, n, inner, device=dev, generator=g).to(torch.bfloat16)
    k = torch.randn(R, nk, inner, device=dev, generator=g).to(torch.bfloat16)
    v = torch.randn(R, nk, inner, device=dev, generator=g).to(torch.bfloat16)
    ctx = torch.empty(R, heads, 64, 64, dtype=torch.bfloat16, device=dev)
    o = torch.empty_like(q)
    # cosine-sim inputs: unit rows, q pre-scaled by 8 log2(e) as the to_q epilogue leaves them
    qc = (F.normalize(q.float().view(R, n, heads, 64), dim=-1) * 8 * LOG2E).view(R, n, inner).to(torch.bfloat16)
    kc = F.normalize(k.float().view(R, nk, heads, 64), dim=-1).view(R, nk, inner).to(torch.bfloat16)
    calls = {
        'context (b200_linear_xattn_context)': lambda: lib.b200_linear_xattn_context(k.data_ptr(), v.data_ptr(), nk * inner, inner, nk, R, heads, 64,
                                                                                      ctx.data_ptr(), st),
        'linear (linear_cross_attn_tc_kernel)': lambda: lib.b200_linear_cross_attention(q.data_ptr(), o.data_ptr(), n * inner, inner, n, ctx.data_ptr(),
                                                                                         R, heads, 64, st),
        'cosine-sim (b200_attention -> cross_attn_tc_kernel)': lambda: lib.b200_attention(qc.data_ptr(), o.data_ptr(), n * inner, 64, inner, n, kc.data_ptr(),
                                                                                           v.data_ptr(), nk * inner, 64, inner, nk, R, heads,
                                                                                           8 * LOG2E * 1.02, st),
    }
    for name, fn in calls.items():                     # warm-up: module load, smem opt-in, tensor-map encode
        for _ in range(5):
            _lib.check(fn(), name)
    torch.cuda.synchronize(dev)
    times = {name: [] for name in calls}
    for _ in range(rounds):                            # alternate the kernels: host noise hits all of them alike
        for name, fn in calls.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                fn()
            e1.record()
            torch.cuda.synchronize(dev)
            times[name].append(e0.elapsed_time(e1) * 1e3 / iters)
    qo_bytes = 2 * R * n * inner * 2
    lines = [f'kernel time, R={R} rows x {n} pixels, {heads} x 64 heads, {nk} keys; {rounds} alternated rounds of {iters} launches each',
             f'q + o traffic {qo_bytes / 1e6:.0f} MB per attention launch; copy rate {COPY_GBS:.0f} GB/s',
             f'{"kernel":<55} {"min us":>9} {"median us":>10} {"max us":>9} {"q+o GB/s":>9} {"of copy":>8}']
    for name, ts in times.items():
        ts = sorted(ts)
        med = ts[len(ts) // 2]
        if name.startswith('context'):
            gbs = 2 * R * nk * inner * 2 / (med * 1e-6) / 1e9
            lines.append(f'{name:<55} {ts[0]:9.1f} {med:10.1f} {ts[-1]:9.1f} {"(k+v " + format(gbs, ".0f") + ")":>9} {"":>8}')
        else:
            gbs = qo_bytes / (med * 1e-6) / 1e9
            lines.append(f'{name:<55} {ts[0]:9.1f} {med:10.1f} {ts[-1]:9.1f} {gbs:9.0f} {gbs / COPY_GBS:8.1%}')
    return lines


def whole_step(dev, steps=100, bs=16, rounds=3):
    models = {}
    for lin in (False, True):
        torch.manual_seed(0)
        u = b2.Unet(dim=128, use_linear_cross_attn=lin)
        with torch.no_grad():
            u.final_conv.weight.normal_(0, 0.02)
            u.final_conv.bias.normal_(0, 0.02)
        models[lin] = b2.Imagen(u, image_sizes=64, timesteps=steps).to(dev)
    te = torch.randn(bs, 256, 768, device=dev)
    res = {lin: [] for lin in models}
    launches = {}
    for lin, im in models.items():                     # warm-up: plan build, graph capture
        im.sample(text_embeds=te, cond_scale=3., use_tqdm=False)
    for _ in range(rounds):
        for lin, im in models.items():
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            im.sample(text_embeds=te, cond_scale=3., use_tqdm=False)
            e1.record()
            torch.cuda.synchronize(dev)
            res[lin].append(e0.elapsed_time(e1) / steps)
            launches[lin] = im.last_launch_count / steps
    lines = [f'whole step: Unet(dim=128) 64x64, bs={bs} with CFG (R={2 * bs}), cond_scale 3, {steps} DDPM steps per sample() call '
             f'(per-call conditioning included), {rounds} alternated calls each']
    for lin in models:
        lines.append(f'  use_linear_cross_attn={str(lin):<5}  ms/step ' + ' '.join(f'{t:.3f}' for t in res[lin]) +
                     f'   launches/step {launches[lin]:.0f}')
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'needs a B200'
    dev = torch.device('cuda', 0)
    _lib.require_device(0)
    lines = [f'GPU: {gpu_info()} (name, power limit, max SM clock; read in this run)']
    lines += kernels(dev)
    lines += whole_step(dev)
    lines.append(f'GPU after the run: {gpu_info()}')
    text = '\n'.join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
