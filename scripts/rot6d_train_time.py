"""Time the 63-D (axis-angle) and 126-D (rot6d) score networks' training step and likelihood function evaluation on one
GPU, in one process, alternating the two widths:

    python scripts/rot6d_train_time.py [--reps 5] [--steps 20] [--out results.jsonl]

Cases: the training step (loss + backward + clip + Adam + EMA) eager and as a CUDA graph at B = 1280 and 16 384, and one
likelihood function evaluation (time table + dpb_score_jvp + dpb_pf_ode_rhs_dim) at 16 384 rows.  Every case is warmed
up, then timed with CUDA events over --steps calls; --reps rounds alternate the widths and the median is reported.
Prints the GPU name and power limit first (nvidia-smi, query only)."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dposer_b200 import losses, ode, sde_lib, synthetic  # noqa: E402
from dposer_b200.ema import ExponentialMovingAverage  # noqa: E402


def gpu_info():
    try:
        return subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0) + ', power limit unknown'


def train_case(pose_dim, B, graph):
    cfg = synthetic.default_config()
    cfg.optim.warmup = 0
    model = synthetic.make_score_model(42, pose_dim=pose_dim).cuda()
    model.train()
    state = dict(optimizer=losses.get_optimizer(cfg, model.parameters()), model=model, step=0,
                 ema=ExponentialMovingAverage(model.parameters(), decay=cfg.model.ema_rate))
    step_fn = losses.get_step_fn(sde_lib.subVPSDE(0.1, 20., 1000), True, losses.optimization_manager(cfg),
                                 reduce_mean=True, graph=graph)
    data = torch.randn(B, model.pose_width, generator=torch.Generator().manual_seed(B)).cuda() * 0.8
    return lambda: step_fn(state, data)


def likelihood_case(pose_dim, B):
    model = synthetic.make_score_model(42, pose_dim=pose_dim).cuda()
    gen = torch.Generator().manual_seed(B)
    x = torch.randn(B, model.pose_width, generator=gen).cuda()
    eps = (torch.randint(0, 2, (B, model.pose_width), generator=gen).float() * 2 - 1).cuda()
    be = ode.PFOdeBackend(model, sde_lib.subVPSDE(0.1, 20., 1000), x, eps)
    return lambda: be._f(0.5, 1)


def time_ms(fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--out')
    a = ap.parse_args()
    assert torch.cuda.is_available(), 'needs a CUDA device'
    info = gpu_info()
    print(f'# GPU: {info}', flush=True)
    cases = [('train_eager', 1280), ('train_graph', 1280), ('train_eager', 16384), ('train_graph', 16384),
             ('likelihood_eval', 16384)]
    results = []
    for name, B in cases:
        fns = {}
        for pd in (3, 6):
            fns[pd] = (likelihood_case(pd, B) if name == 'likelihood_eval' else
                       train_case(pd, B, graph=name == 'train_graph'))
            for _ in range(a.warmup):
                fns[pd]()
        torch.cuda.synchronize()
        times = {3: [], 6: []}
        for _ in range(a.reps):
            for pd in (3, 6):
                times[pd].append(time_ms(fns[pd], a.steps))
        m63, m126 = statistics.median(times[3]), statistics.median(times[6])
        r = dict(case=name, B=B, ms_63=round(m63, 4), ms_126=round(m126, 4), ratio=round(m126 / m63, 4),
                 spread_63=[round(min(times[3]), 4), round(max(times[3]), 4)],
                 spread_126=[round(min(times[6]), 4), round(max(times[6]), 4)], gpu=info)
        print(json.dumps(r), flush=True)
        results.append(r)
        del fns
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, 'w') as f:
            for r in results:
                f.write(json.dumps(r) + '\n')


if __name__ == '__main__':
    main()
