"""Time the 63-D (axis) and 126-D (rot6d) score networks on the tcgen05 engine at 65 536 rows: one forward pass, the
1000-step Euler-Maruyama sampler and the prior loss.  Prints one JSON line per (width, workload) with the median of
--reps timed calls (CUDA events; the two widths alternate call by call) and the achieved rate at

    63-D:  8 646 656 FLOP per row per network evaluation   (2 * 1024 * (63 + 4 * 1024 + 63))
    126-D: 8 904 704 FLOP per row per network evaluation   (2 * 1024 * (126 + 4 * 1024 + 126))

against the bf16 dense rate this GPU sustains on a large torch.matmul measured in the same run (the roof the kernel's
fp16 / bf16 tensor-core MMAs share).  The first line records the GPU, its power limit and clocks.

    python scripts/rot6d_time.py [--rows 65536] [--steps 1000] [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dposer_b200 import _lib as L  # noqa: E402
from dposer_b200 import prior, sampling, sde_lib, synthetic  # noqa: E402

FLOP_PER_ROW = {63: 2 * 1024 * (63 + 4 * 1024 + 63), 126: 2 * 1024 * (126 + 4 * 1024 + 126)}


def gpu_info():
    q = 'name,power.limit,clocks.sm,clocks.max.sm,clocks.mem,temperature.gpu'
    try:
        out = subprocess.run(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader', '-i', '0'],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:      # noqa: BLE001
        out = f'unavailable: {e}'
    return dict(zip(q.split(','), [s.strip() for s in out.split(',')]))


def timed(fn, reps):
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b) / 1e3)
    return sorted(ts)[len(ts) // 2]


def bf16_peak(reps=20, n=8192):
    a = torch.randn(n, n, device='cuda', dtype=torch.bfloat16)
    b = torch.randn(n, n, device='cuda', dtype=torch.bfloat16)
    for _ in range(3):
        a @ b

    def run():
        for _ in range(reps):
            a @ b
    t = timed(run, 5)
    return 2 * n ** 3 * reps / t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rows', type=int, default=65536)
    ap.add_argument('--steps', type=int, default=1000)
    ap.add_argument('--reps', type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('rot6d_time.py measures on the GPU: no CUDA device')
    B, N = args.rows, args.steps
    print(json.dumps({'gpu': gpu_info()}), flush=True)
    peak = bf16_peak()
    print(json.dumps({'bf16_matmul_tflops': peak / 1e12}), flush=True)
    cfg = synthetic.default_config()
    sde = sde_lib.subVPSDE(0.1, 20., N)
    gen = torch.Generator().manual_seed(0)
    runs = {}
    for pd, D in ((3, 63), (6, 126)):
        m = synthetic.make_score_model(42, pose_dim=pd).cuda()
        m.engine = L.ENGINE_TC
        x = torch.randn(B, D, generator=gen).cuda()
        out = torch.empty_like(x)
        table = m.time_table(torch.full((1,), 500.0))         # built once: the timed forward is the network alone
        ws = m.workspace(B, x.device)
        fn = sampling.get_sampling_fn(cfg, sde, (B, D), lambda v: v, 1e-3, device='cuda', return_trajs=False)
        comp = prior.DPoserComp(m, sde_lib.subVPSDE(0.1, 20., 1000), True, batch_size=B)

        def forward(m=m, x=x, out=out, table=table, ws=ws):
            L.check(L.load().dpb_score_forward(m.handle().ptr, L.ptr(x), L.ptr(table), None, None, 1.0, L.ptr(out), B,
                                               L.ENGINE_TC, L.ptr(ws), ws.numel(), L.current_stream(x.device)))
        runs[D] = {
            'forward': (forward, 1),
            'sampler': (lambda m=m, fn=fn, x=x: fn(m, z=x), N),
            'prior_loss': (lambda comp=comp, x=x: comp.loss(x, 0.5), 1),   # host float t: no device read in the window
        }
        for f, _ in runs[D].values():
            f()
        torch.cuda.synchronize()
    for name in ('forward', 'sampler', 'prior_loss'):
        times = {63: [], 126: []}
        for _ in range(args.reps):                     # alternate the widths call by call
            for D in (63, 126):
                times[D].append(timed(runs[D][name][0], 1))
        for D in (63, 126):
            t = sorted(times[D])[len(times[D]) // 2]
            flop = FLOP_PER_ROW[D] * B * runs[D][name][1]
            print(json.dumps({'width': D, 'workload': name, 'rows': B, 'evals_per_row': runs[D][name][1],
                              'seconds_median': t, 'seconds_all': times[D], 'tflops': flop / t / 1e12,
                              'fraction_of_bf16_matmul': flop / t / peak}), flush=True)
    print(json.dumps({'gpu_after': gpu_info()}), flush=True)


if __name__ == '__main__':
    main()
