"""Time the native fitting chains with a 63-D (axis) and a 126-D (rot6d) DPoser prior, and the two axis -> rot6d
kernels alone.  Prints one JSON line per measurement; the first line records the GPU and its power limit.

* c5 SMPLify shard: 131 072 images, 100 camera + 5 x 100 body Adam steps (bench.py's configs[4] problem), plain
  launches as bench.py runs it; the two priors alternate run by run.  One further run per prior with graphs=True
  checks that the captured chain is finite at this size.
* c4 motion denoising: batches of 256 x 60 frames, 3 x 60 Adam steps, CUDA graphs captured by a first batch and
  replayed by the timed ones (bench.py's configs[3]); the priors alternate batch by batch.
* dpb_axis_to_rot6d_cols and its VJP at 15 360 and 131 072 rows (x strided as SMPL-X's full_pose, ld 165): CUDA events
  around --launches back-to-back launches; bytes moved against the 6 551.7 GB/s HBM copy rate of BASELINE.md.

    python scripts/rot6d_fit_time.py [--images 131072] [--sequences 256] [--batches 4] [--reps 2] [--launches 2000]
"""
import argparse
import json
import os
import sys
import time
import types

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dposer_b200 import fitting, prior, sde_lib, steps, synthetic  # noqa: E402
from dposer_b200.body_model import BodyModel, SMPLX  # noqa: E402
from dposer_b200.misc import Posenormalizer  # noqa: E402
from scripts.rot6d_time import gpu_info  # noqa: E402

COPY_GBS = 6551.7


def emit(**kw):
    print(json.dumps(kw), flush=True)


def priors():
    """(name, model, normaliser) of the two widths: the same synthetic recipe, seed 42."""
    out = []
    for name, pd, rep in (('axis', 3, 'axis'), ('rot6d', 6, 'rot6d')):
        out.append((name, synthetic.make_score_model(42, pose_dim=pd).cuda(),
                    Posenormalizer(None, device='cuda', normalize=True, min_max=False, rot_rep=rep)))
    return out


def kernel_times(launches):
    for rows in (15360, 131072):
        full = torch.randn(rows, 165, device='cuda') * 0.5
        mean, std = (t.float().contiguous() for t in
                     Posenormalizer(None, device='cuda', min_max=False, rot_rep='rot6d').column_affine())
        x0, g, gx = torch.empty(rows, 126, device='cuda'), torch.randn(rows, 126, device='cuda'), \
            torch.empty(rows, 63, device='cuda')
        calls = {'forward': (lambda: steps.axis_to_rot6d_cols(full, 3, mean, std, x0), rows * (63 + 126) * 4),
                 'vjp': (lambda: steps.axis_to_rot6d_cols_vjp(full, 3, std, g, gx), rows * (63 + 126 + 63) * 4)}
        for name, (fn, nbytes) in calls.items():
            for _ in range(20):
                fn()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(launches):
                fn()
            b.record()
            b.synchronize()
            s = a.elapsed_time(b) / 1e3 / launches
            emit(kernel=name, rows=rows, launches=launches, us=s * 1e6, mbytes=nbytes / 1e6,
                 gbs=nbytes / s / 1e9, fraction_of_copy_rate=nbytes / s / 1e9 / COPY_GBS,
                 note='back-to-back launches; the working set fits the 126 MB L2 at 15 360 rows')


def c5(models, images, reps):
    dev = torch.device('cuda')
    mx = synthetic.make_body_tensors('smplx')
    B = images
    smpl = SMPLX(mx, batch_size=B).to(dev)
    g = torch.Generator().manual_seed(41)
    body = synthetic.toy_poses().repeat((B + 499) // 500, 1)[:B]
    glob = torch.tensor([3.14159, 0., 0.]) + 0.2 * torch.randn(B, 3, generator=g)
    cam = torch.stack([0.2 * torch.randn(B, generator=g), 0.2 * torch.randn(B, generator=g),
                       20 + 20 * torch.rand(B, generator=g)], 1)
    betas = torch.randn(B, 10, generator=g)
    with torch.no_grad():
        j = smpl(betas=betas.to(dev), body_pose=body.to(dev), global_orient=glob.to(dev), transl=cam.to(dev)).joints
        center = torch.full((B, 2), 512., device=dev)
        kp = torch.stack([5000 * j[..., 0] / j[..., 2] + 512, 5000 * j[..., 1] / j[..., 2] + 512], -1) + \
            2 * torch.randn(B, 49, 2, device=dev)
        conf = 0.3 + 0.7 * torch.rand(B, 49, device=dev)
        conf[:, 25:] = 0
        kp2d = torch.cat([kp, conf[..., None]], -1)
    sargs = types.SimpleNamespace(device=dev, sde_N=500, time_strategy='3')
    init_pose = torch.cat([glob + 0.1, smpl.mean_poses[3:66].cpu()[None].repeat(B, 1)], 1).to(dev)
    init_betas = smpl.mean_shape[None].repeat(B, 1).to(dev)
    init_cam = (cam + torch.tensor([0.1, -0.1, 2.0])).to(dev)
    fits = {}
    for name, model, norm in models:
        pp = prior.DPoser(batch_size=B, args=sargs, model=model, sde=sde_lib.subVPSDE(0.1, 20., 1000), normalizer=norm)
        fitting.SMPLify(smpl, step_size=1e-2, batch_size=B, num_iters=2, focal_length=5000., args=sargs,
                        pose_prior=pp)(init_pose, init_betas, init_cam, center, kp2d.clone())     # warm-up
        fits[name] = fitting.SMPLify(smpl, step_size=1e-2, batch_size=B, num_iters=100, focal_length=5000., args=sargs,
                                     pose_prior=pp)
    torch.cuda.synchronize()
    times = {name: [] for name in fits}
    finite = {name: True for name in fits}
    for _ in range(reps):
        for name, fit in fits.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pose, _, _, reproj = fit(init_pose, init_betas, init_cam, center, kp2d.clone())
            torch.cuda.synchronize()
            times[name].append(time.perf_counter() - t0)
            finite[name] = finite[name] and bool(torch.isfinite(pose).all() and torch.isfinite(reproj).all())
    for name in fits:
        t = min(times[name])
        emit(config='c5_smplify', prior=name, images=B, adam_steps=600, graphs=False, seconds_all=times[name],
             ms_per_adam_step=t * 1e3 / 600, finite=finite[name])
    for name, fit in fits.items():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pose, _, _, reproj = fit(init_pose, init_betas, init_cam, center, kp2d.clone(), graphs=True)
        torch.cuda.synchronize()
        emit(config='c5_smplify', prior=name, images=B, adam_steps=600, graphs=True,
             seconds_including_capture=time.perf_counter() - t0,
             finite=bool(torch.isfinite(pose).all() and torch.isfinite(reproj).all()))
    del fits, smpl
    torch.cuda.empty_cache()


def c4(models, n_seq, batches):
    dev = torch.device('cuda')
    Lf = 60
    rows = n_seq * Lf
    mx = synthetic.make_body_tensors('smplx')
    bm = BodyModel(mx, num_betas=10, batch_size=rows, model_type='smplx').to(dev)
    ges, _ = synthetic.gesture_sequences()
    gt = ges[:Lf].repeat(n_seq, 1).to(dev)
    with torch.no_grad():
        jn = bm(pose_body=gt, need_verts=False).Jtr[:, :22] + 0.04 * torch.randn(rows, 22, 3, device=dev)
    kw = dict(time_strategy='3', sample_trun=4.0, sample_time=490, iterations=3, steps_per_iter=60, graphs=True)
    mds = {}
    for name, model, norm in models:
        mds[name] = fitting.MotionDenoise(synthetic.default_config(), types.SimpleNamespace(device=dev), model, bm,
                                          sde_lib.subVPSDE(0.1, 20., 1000), norm, sde_N=500, batch_size=rows,
                                          seq_len=Lf)
        mds[name].optimize(jn, **kw)              # first batch: allocates, captures the 180 step graphs
    torch.cuda.synchronize()
    times = {name: [] for name in mds}
    finite = {name: True for name in mds}
    for _ in range(batches):
        for name, md in mds.items():
            md.poses = torch.randn(rows, 63, device=dev) * 0.01
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = md.optimize(jn, gt_poses=None, **kw)
            torch.cuda.synchronize()
            times[name].append(time.perf_counter() - t0)
            finite[name] = finite[name] and bool(torch.isfinite(res['pose_body']).all())
    for name in mds:
        t = sorted(times[name])[len(times[name]) // 2]
        emit(config='c4_motion_denoise', prior=name, frames_per_batch=rows, batches=batches, adam_steps=180,
             graphs=True, seconds_all=times[name], ms_per_adam_step=t * 1e3 / 180, finite=finite[name])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--images', type=int, default=131072)
    ap.add_argument('--sequences', type=int, default=256)
    ap.add_argument('--batches', type=int, default=4)
    ap.add_argument('--reps', type=int, default=2)
    ap.add_argument('--launches', type=int, default=2000)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('rot6d_fit_time.py measures on the GPU: no CUDA device')
    emit(gpu=gpu_info())
    kernel_times(args.launches)
    models = priors()
    c4(models, args.sequences, args.batches)
    c5(models, args.images, args.reps)
    emit(gpu_after=gpu_info())


if __name__ == '__main__':
    main()
