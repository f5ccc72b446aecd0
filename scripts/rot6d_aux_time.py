"""Time the rot6d -> axis-angle kernels of the auxiliary training loss and the auxiliary step itself at both widths.
Prints one JSON line per measurement; the first line records the GPU and its power limit.

* dpb_rot6d_to_axis_cols and its VJP (x [rows, 126] contiguous, 21 joints) at --rows: CUDA events around --launches
  back-to-back launches.  Bytes per row: forward 756 (504 in, 252 out), VJP 1260 (504 + 252 in, 504 out), against the
  device-to-device copy rate measured in the same run.  At 131 072 rows the forward's working set (99 MB) fits the
  126 MB L2; 1 048 576 rows do not.
* get_step_fn(auxiliary_loss=True) at the reference configuration (batch 1280, 10 denoise steps, SMPL-X with all
  vertices; scripts/train_aux_time.py's setup) for a 63-D network (rot_rep='axis') and a 126-D one (rot_rep='rot6d'),
  alternating round by round in one process: CUDA events over --steps steps after 3 warm-up steps, median of --rounds.

    python scripts/rot6d_aux_time.py [--rows 131072,1048576] [--launches 2000] [--batch 1280] [--denoise 10]
                                     [--steps 10] [--rounds 5]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dposer_b200 import losses, sde_lib, steps, synthetic  # noqa: E402
from dposer_b200.body_model import BodyModel  # noqa: E402
from dposer_b200.ema import ExponentialMovingAverage  # noqa: E402
from dposer_b200.misc import Posenormalizer  # noqa: E402
from scripts.rot6d_time import gpu_info  # noqa: E402


def emit(**kw):
    print(json.dumps(kw), flush=True)


def events(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3 / n


def copy_rate():
    src = torch.empty(1 << 28, device='cuda')          # 1 GiB
    dst = torch.empty_like(src)
    for _ in range(5):
        dst.copy_(src)
    s = events(lambda: dst.copy_(src), 50)
    gbs = 2 * src.numel() * 4 / s / 1e9
    emit(measurement='device copy', gib=1, gbs=gbs)
    return gbs


def kernel_times(rows_list, launches, copy_gbs):
    mean, std = (t.float().contiguous() for t in
                 Posenormalizer(None, device='cuda', min_max=False, rot_rep='rot6d').column_affine())
    for rows in rows_list:
        x = torch.randn(rows, 126, device='cuda')
        out, g, gx = torch.empty(rows, 63, device='cuda'), torch.randn(rows, 63, device='cuda'), \
            torch.empty(rows, 126, device='cuda')
        calls = {'forward': (lambda: steps.rot6d_to_axis_cols(x, 0, mean, std, out), rows * 756),
                 'vjp': (lambda: steps.rot6d_to_axis_cols_vjp(x, 0, mean, std, g, gx), rows * 1260)}
        for name, (fn, nbytes) in calls.items():
            for _ in range(20):
                fn()
            s = events(fn, launches)
            emit(kernel=name, rows=rows, launches=launches, us=s * 1e6, mbytes=nbytes / 1e6, gbs=nbytes / s / 1e9,
                 fraction_of_copy_rate=nbytes / s / 1e9 / copy_gbs, note='back-to-back launches')


def aux_steps(B, N, n_steps, rounds):
    cfg = synthetic.default_config()
    bm = BodyModel(synthetic.make_body_tensors('smplx'), num_betas=10, batch_size=B, model_type='smplx').cuda()
    toy = synthetic.toy_poses()
    idx = torch.randint(0, toy.shape[0], (B,), generator=torch.Generator().manual_seed(0))
    runs = {}
    for width, pd, rep in ((63, 3, 'axis'), (126, 6, 'rot6d')):
        model = synthetic.make_score_model(42, pose_dim=pd).cuda()
        model.train()
        norm = Posenormalizer(None, device='cuda', normalize=True, min_max=False, rot_rep=rep)
        state = dict(optimizer=losses.get_optimizer(cfg, model.parameters()), model=model,
                     ema=ExponentialMovingAverage(model.parameters(), decay=cfg.model.ema_rate), step=0)
        fn = losses.get_step_fn(sde_lib.subVPSDE(0.1, 20., 1000), True, losses.optimization_manager(cfg),
                                reduce_mean=True, auxiliary_loss=True, denormalize=norm.offline_denormalize,
                                body_model=bm, rot_rep=rep, denoise_steps=N)
        data = norm.offline_normalize(toy[idx].cuda(), from_axis=rep == 'rot6d')
        for _ in range(3):
            ld = fn(state, data)
        runs[width] = (fn, state, data)
    times = {63: [], 126: []}
    for _ in range(rounds):
        for width, (fn, state, data) in runs.items():
            times[width].append(events(lambda: fn(state, data), n_steps) * 1e3)
    med = {w: sorted(t)[len(t) // 2] for w, t in times.items()}
    for w in (63, 126):
        emit(measurement='auxiliary step', width=w, batch=B, denoise_steps=N, ms_per_step=med[w], rounds=times[w])
    emit(measurement='auxiliary step ratio', ratio_126_over_63=med[126] / med[63])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rows', default='131072,1048576')
    ap.add_argument('--launches', type=int, default=2000)
    ap.add_argument('--batch', type=int, default=1280)
    ap.add_argument('--denoise', type=int, default=10)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--rounds', type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('rot6d_aux_time.py measures on a CUDA device; none is visible')
    emit(gpu=gpu_info())
    kernel_times([int(r) for r in a.rows.split(',')], a.launches, copy_rate())
    aux_steps(a.batch, a.denoise, a.steps, a.rounds)


if __name__ == '__main__':
    main()
