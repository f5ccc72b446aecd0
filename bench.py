#!/usr/bin/env python
"""Benchmark of the DPoser hot path: poses/sec for reverse-SDE sampling + SMPL LBS.

    python bench.py --gpus N --steps K --warmup W [--workload sample_lbs|lbs|sample|completion] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic input resident in HBM:
  sample_lbs (default): x_T[B,63] -> 1000-step reverse SDE (EM predictor, subVP, config default) ->
                        de-normalise -> SMPL LBS forward (6890 verts / 45 joints).  B = 65536 per GPU
                        (BASELINE.json configs[1] batch; the metric "reverse-SDE sampling + SMPL LBS").
  lbs:     configs[1] alone (SMPL LBS forward, B = 65536).
  sample:  the sampler alone.     completion: configs[2] (imputation sampler, 40960 rows).
Prints ONE JSON line (rank 0).  `--dump-outputs DIR` also writes what the last timed step returned (rank 0) as
float32 DIR/<name>.npy; all inputs are seeded, so two builds run with the same arguments compare output for output.
Multi-GPU: rows are independent, every rank processes its own B rows
(weak scaling, no data-path collective in `value`); timing is barrier + CUDA events, max over ranks.  The end-to-end
leg (`e2e`) at N > 1 also runs the collectives the reference's evaluation uses (run/completion.py:300-305,
lib/utils/metric.py:8-37): all-gather of the generated poses and the rank-sharded APD with its all-reduce.

Keys beyond the contract:
  roofline          the fused sampler kernel against the measured sustained bf16 peak, with `roofline.lbs` = the LBS
                    forward against the measured HBM copy bandwidth (and against its three-product tensor floor)
  configs           (N = 1) every BASELINE.json config measured at its stated size, or the largest batch of independent
                    problems that is one pass of the path (stated), each with the CPU port's figure
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SCORE_FLOP_PER_ROW = 8646656          # SURVEY 8(d): 2*(63*1024 + 4*1024^2 + 1024*63), batch-uniform t
LBS_BYTES_PER_POSE = 83560            # SURVEY 8(d): verts 6890*12 + joints 45*12 + inputs 85*4
# DRAM traffic from the committed `ncu --set full` capture (profiles/r2_ncu_full_summary.md):
#   fused sampler: 60.5 MB read + 255.7 MB written for 18 944 rows x 4 steps (write-back of the L2-resident activation
#   scratch; 1.201 GB per 37 888 x 4 before the evict_last hints)
#   LBS: lt3::lbs_fused3_kernel 547 MB read + 5.377 GB written for 65 536 poses (profiles/r2_ncu_fused3_l2_hints.md: the
#   output plus operand refills; 1.474 GB read without the L2 hints; 326 MB + 1.311 GB per 16 384 poses before them)
SAMPLER_DRAM_BYTES_PER_ROW_STEP = (60.514e6 + 255.652e6) / (18944 * 4)
LBS_DRAM_BYTES_PER_POSE = (546.978e6 + 5377.018e6) / 65536
# tensor floor of the LBS forward at three fp16 products: (63 blend + 38.4 skinning) tensor-pipe cycles per (pose,
# 128-vertex tile), 54 tiles, 148 SMs, 1.92 GHz (DESIGN.md, LBS design)
LBS_TENSOR_FLOOR_MS = 65536 * 54 * 101.4 / 148 / 1.92e9 * 1e3
N_SDE = 1000


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d['hbm_gbs'], tc_burst=d['bf16_tflops'], tc_sustained=d['bf16_tflops_sustained'],
                    src='measured')
    return dict(hbm=6650.0, tc_burst=1590.0, tc_sustained=1400.0, src='fallback')   # B200_PROFILING.md fallback


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-i', str(self.index), '-lms', '200'], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i] == 'Active' for r in self.rows)]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(sm)}


# ------------------------------------------------------------------------------------------- CPU reference arm
def _reference_sampler(workload, rows):
    """The UNMODIFIED reference sampler (oracle/_ref, staged by oracle/make_ref.py from /root/reference) with the
    synthetic weights recipe, or None when the staged modules are absent."""
    from dposer_b200 import synthetic
    from oracle import make_ref
    mods = make_ref.import_reference()
    if mods is None:
        return None
    model_m, sde_m, _, sampling_m = mods
    cfg = synthetic.default_config()
    cfg.device = torch.device('cpu')
    torch.manual_seed(42)
    model = model_m.ScoreModelFC(cfg, n_poses=21, pose_dim=3, hidden_dim=1024, embed_dim=512, n_blocks=2)
    for mod in model.modules():
        if isinstance(mod, torch.nn.GroupNorm):
            with torch.no_grad():
                mod.weight.copy_(torch.rand(1024) + 0.5)
                mod.bias.copy_(torch.randn(1024) * 0.1)
    model.eval()
    sde = sde_m.subVPSDE(beta_min=0.1, beta_max=20., N=N_SDE)
    fn = sampling_m.get_pc_sampler(sde, (rows, 63), sampling_m.EulerMaruyamaPredictor, sampling_m.NoneCorrector,
                                   lambda x: x, 0.16, n_steps=1, probability_flow=False, continuous=True, denoise=True,
                                   eps=1e-3, device='cpu')
    return model, fn


def cpu_reference(workload, budget_s=20.0):
    """The reference algorithm on the host cores.  Sampler: the reference's own `get_pc_sampler` from oracle/_ref when it
    is staged (kind "reference"), else the oracle port (pinned bit-exactly to it by tests/golden).  LBS: always the port
    (third-party smplx is absent).  Bounded sample, linear in rows (all rows independent)."""
    import types
    from dposer_b200 import synthetic
    from oracle import lbs_ref, score_ref
    cores = os.cpu_count()
    torch.set_num_threads(cores)
    t_pose = 0.0
    sample = []
    kind = 'port'
    if workload in ('sample_lbs', 'sample', 'completion'):
        rows = 256
        gen = torch.Generator().manual_seed(1234)
        x = torch.randn(rows, 63, generator=gen)
        kw = {}
        if workload == 'completion':
            _, mask, obs = synthetic.completion_inputs(n_partial=rows, hypotheses=1)
            kw = dict(observation=obs, mask=mask)
        ref = _reference_sampler(workload, rows)
        if ref is not None:
            kind = 'reference'
            model, fn = ref
            # the stock pc_sampler, all of its steps from `start`: the 'denoise' task is the reference's own way to
            # enter the loop late (sampling.py:451-453); completion keeps its imputation and runs all N steps
            k_steps = max(20, min(N_SDE, int(budget_s * 0.6 / 0.012)))
            if workload == 'completion':
                k_steps, a = N_SDE, types.SimpleNamespace(task='completion')
                t0 = time.perf_counter()
                fn(model, z=x, args=a, **kw)
            else:
                a = types.SimpleNamespace(task='denoise')
                fn(model, z=x, start_step=N_SDE - 3, args=a)                   # warm-up
                t0 = time.perf_counter()
                fn(model, z=x, start_step=N_SDE - k_steps, args=a)
            dt = time.perf_counter() - t0
            t_pose += dt / k_steps * N_SDE / rows
            sample.append(f'reference get_pc_sampler (oracle/_ref, unmodified) on {rows} rows: {k_steps} of {N_SDE} '
                          f'Euler-Maruyama steps in {dt:.1f} s, per-step time x {N_SDE}')
        else:
            sd = score_ref.make_state_dict(42)
            sde = score_ref.SubVP(0.1, 20., N_SDE)
            steps = 8
            if workload == 'completion':
                kw['task'] = 'completion'
            score_ref.pc_sample(sd, sde, x, 1e-3, n_run=1, **kw)                       # warm-up
            t0 = time.perf_counter()
            done = 0
            while time.perf_counter() - t0 < budget_s * 0.6:
                score_ref.pc_sample(sd, sde, x, 1e-3, n_run=steps, **kw)
                done += steps
            dt = time.perf_counter() - t0
            t_pose += dt / done * N_SDE / rows
            sample.append(f'oracle port pc_sampler on {rows} rows: {done} Euler-Maruyama steps timed in runs of {steps}, '
                          f'per-step time x {N_SDE} steps')
    if workload in ('sample_lbs', 'lbs'):
        m = synthetic.make_body_tensors('smpl')
        rows = 512
        inp = synthetic.lbs_inputs(rows, 'smpl')
        pose, shape = synthetic.full_pose_from(inp, 'smpl')
        lbs_ref.body_forward(m, shape[:64], pose[:64], inp['trans'][:64])
        t0 = time.perf_counter()
        done = 0
        while time.perf_counter() - t0 < budget_s * 0.4:
            lbs_ref.body_forward(m, shape, pose, inp['trans'], chunk=256)
            done += rows
        t_pose += (time.perf_counter() - t0) / done
        sample.append(f'SMPL LBS (oracle port of smplx lbs(); smplx itself is not installable here) {done} poses in '
                      'chunks of 256')
    return dict(value=1.0 / t_pose, unit='poses/s', cores=cores, kind=kind, sample='; '.join(sample))


def run_reference_arm(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    t0 = time.perf_counter()
    vals = []
    for _ in range(max(1, args.warmup)):
        cpu_reference(args.workload, budget_s=4.0)
    for _ in range(args.steps):
        vals.append(cpu_reference(args.workload, budget_s=12.0))
    v = sum(x['value'] for x in vals) / len(vals)
    base = vals[-1]
    base['value'] = v
    B = default_batch(args)
    line = {'impl': 'reference', 'metric': 'poses/sec: DPoser reverse-SDE sampling + SMPL LBS', 'value': v,
            'unit': 'poses/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': 1000.0 * B / v, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic', 'config': workload_config(args, B),
            'cpu_baseline': base,
            'e2e': {'value': v, 'unit': 'poses/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0, 'wall_s': time.perf_counter() - t0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------- GPU arm
def default_batch(args):
    if args.batch:
        return args.batch
    return 40960 if args.workload == 'completion' else 65536


def workload_config(args, B):
    names = {'sample_lbs': f'reverse-SDE sampling (subVP, EM predictor, N={args.sde_steps}, eps=1e-3, config default) of '
                           f'{B} poses/GPU + SMPL LBS forward (6890 verts, 24+21 joints, 10 betas) = configs[0] '
                           'pipeline at configs[1] batch',
             'lbs': f'configs[1]: SMPL LBS forward only, batch {B}/GPU',
             'sample': f'reverse-SDE sampling only, N={args.sde_steps}, {B} poses/GPU',
             'completion': f'configs[2]: completion by imputation sampler, {B} rows/GPU, N={args.sde_steps}'}
    return {'workload': names[args.workload], 'batch_per_gpu': B, 'sde_steps': args.sde_steps,
            'l2': 'L2 flushed (256 MiB write) between timed steps', 'engine': args.engine,
            'weights': 'random-init ScoreModelFC (seed 42), synthetic SMPL tensors (seed 7)'}


def _ev_time(f, flush, reps=3):
    """best-of-`reps` CUDA-event time (ms) of f() with the L2 flushed before every run"""
    f()
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(reps):
        flush.fill_(1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        f()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best


def bench_configs(args, dev, model, peaks, flush, cpu_per_row_step):
    """Every BASELINE.json config at its stated size (or one batch of independent problems, stated) on ONE GPU."""
    import types
    from dposer_b200 import _lib as L
    from dposer_b200 import fitting, prior, sampling, sde_lib, synthetic
    from dposer_b200.body_model import BodyModel, SMPLX
    from dposer_b200.misc import Posenormalizer
    out = {}
    cfg = synthetic.default_config()
    norm = Posenormalizer(None, device=dev, normalize=True, min_max=False, rot_rep='axis')
    sde = sde_lib.subVPSDE(0.1, 20., N_SDE)

    def cpu_sampler(evals_per_step=1):
        if cpu_per_row_step is None:
            return None
        return {'value': 1.0 / (cpu_per_row_step * N_SDE * evals_per_step), 'unit': 'poses/s',
                'note': 'CPU arm of this run (cpu_baseline), per row and score evaluation'}

    with torch.no_grad():
        # ---- configs[0] literal: 500 poses, EM predictor (run/demo.py:127-136) and EM + Langevin (--metrics, :137-145)
        B = 500
        z = torch.randn(B, 63, generator=torch.Generator().manual_seed(5)).to(dev)
        fn = sampling.get_sampling_fn(cfg, sde, (B, 63), lambda x: x, 1e-3, device=dev, return_trajs=False)
        ms = _ev_time(lambda: fn(model, z=z), flush)
        tf = SCORE_FLOP_PER_ROW * B * N_SDE / (ms * 1e-3) / 1e12
        out['c1_generation_500_em'] = {
            'workload': 'configs[0] literal: 500 poses, subVP reverse SDE, N=1000, EM predictor', 'rows': B, 'ms': ms,
            'value': B / (ms * 1e-3), 'unit': 'poses/s', 'ms_per_sde_step': ms / N_SDE,
            'roofline': {'bound': 'latency (4 row tiles on 148 SMs)', 'achieved': tf, 'unit': 'TFLOP/s',
                         'frac_of_tensor_peak': tf / peaks['tc_sustained']}, 'cpu': cpu_sampler()}
        cfg_l = synthetic.default_config()
        cfg_l.sampling.corrector = 'langevin'
        fn_l = sampling.get_sampling_fn(cfg_l, sde, (B, 63), lambda x: x, 1e-3, device=dev, return_trajs=False)
        ms = _ev_time(lambda: fn_l(model, z=z), flush, reps=2)
        out['c1_generation_500_pc'] = {
            'workload': 'configs[0] --metrics variant: EM predictor + Langevin corrector (snr 0.16), 2 score '
                        'evaluations per step', 'rows': B, 'ms': ms, 'value': B / (ms * 1e-3), 'unit': 'poses/s',
            'ms_per_sde_step': ms / N_SDE, 'cpu': cpu_sampler(2)}

        # ---- configs[2]: completion by imputation sampler, 10 hypotheses x 4096 partial poses
        B = 40960
        _, mask, obs = synthetic.completion_inputs(n_partial=B // 10, hypotheses=10, seed=21)
        mask, obs = mask.to(dev), obs.to(dev)
        z = torch.randn(B, 63, generator=torch.Generator().manual_seed(6)).to(dev)
        fn_c = sampling.get_sampling_fn(cfg, sde, (B, 63), lambda x: x, 1e-3, device=dev, return_trajs=False)
        targs = types.SimpleNamespace(task='completion')
        ms = _ev_time(lambda: fn_c(model, z=z, observation=obs, mask=mask, args=targs), flush, reps=2)
        tf = SCORE_FLOP_PER_ROW * B * N_SDE / (ms * 1e-3) / 1e12
        out['c3_completion'] = {
            'workload': 'configs[2]: 10 hypotheses x 4096 partial poses (legs masked), imputation sampler, N=1000',
            'rows': B, 'ms': ms, 'value': B / (ms * 1e-3), 'unit': 'poses/s',
            'roofline': {'bound': 'tensor', 'achieved': tf, 'peak': peaks['tc_sustained'], 'unit': 'TFLOP/s',
                         'frac': tf / peaks['tc_sustained']}, 'cpu': cpu_sampler()}
        del mask, obs, z

    # ---- configs[3]: motion denoising, SMPL-X, 3 x 60 Adam steps (run/motion_denoising.py:332), batches of sequences
    n_seq, Lf = args.c4_sequences, 60
    rows = n_seq * Lf
    mx = synthetic.make_body_tensors('smplx')
    bm = BodyModel(mx, num_betas=10, batch_size=rows, model_type='smplx').to(dev)
    ges, _ = synthetic.gesture_sequences()
    gt = ges[:Lf].repeat(n_seq, 1).to(dev)
    with torch.no_grad():
        jn = bm(pose_body=gt, need_verts=False).Jtr[:, :22] + 0.04 * torch.randn(rows, 22, 3, device=dev)
    md = fitting.MotionDenoise(cfg, types.SimpleNamespace(device=dev), model, bm, sde_lib.subVPSDE(0.1, 20., N_SDE), norm,
                               sde_N=500, batch_size=rows, seq_len=Lf)
    kw = dict(time_strategy='3', sample_trun=4.0, sample_time=490, iterations=3, steps_per_iter=60, graphs=True)
    md.optimize(jn, **kw)                      # first batch: allocates, captures the 180 step graphs
    torch.cuda.synchronize()
    n_batches = args.c4_batches if args.c4_batches > 0 else max(1, 8192 // n_seq)
    flush.fill_(1)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    finite = True
    for _ in range(n_batches):                 # further batches of sequences: graph replays only
        md.poses = torch.randn(rows, 63, device=dev) * 0.01
        res = md.optimize(jn, gt_poses=None, **kw)
        finite = finite and bool(torch.isfinite(res['pose_body']).all())
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    out['c4_motion_denoise'] = {
        'workload': f'configs[3]: DPoser prior + temporal vertex term + joint data term, SMPL-X (10475 verts), Adam 3 x 60 '
                    f'steps; {n_batches * n_seq} independent 60-frame sequences as {n_batches} batches of {n_seq} replaying '
                    'the same captured step graphs (vertices + cotangents of one batch: 3.9 GB)',
        'sequences': n_batches * n_seq, 'frames': n_batches * rows, 'adam_steps': 180, 'seconds': dt,
        'value': n_batches * rows / dt, 'unit': 'frames/s', 'ms_per_adam_step': dt * 1e3 / (180 * n_batches),
        'frames_per_batch': rows, 'finite': finite}
    del md, bm, jn, gt, res
    torch.cuda.empty_cache()

    # ---- configs[4]: SMPLify, SMPL-X joints, 100 camera + 5 x 100 body Adam steps (run/fitting.py:117), per-GPU shard
    B = args.c5_images
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
    pp = prior.DPoser(batch_size=B, args=sargs, model=model, sde=sde_lib.subVPSDE(0.1, 20., N_SDE), normalizer=norm)
    init_pose = torch.cat([glob + 0.1, smpl.mean_poses[3:66].cpu()[None].repeat(B, 1)], 1).to(dev)
    init_betas = smpl.mean_shape[None].repeat(B, 1).to(dev)
    init_cam = (cam + torch.tensor([0.1, -0.1, 2.0])).to(dev)
    warm = fitting.SMPLify(smpl, step_size=1e-2, batch_size=B, num_iters=2, focal_length=5000., args=sargs, pose_prior=pp)
    warm(init_pose, init_betas, init_cam, center, kp2d.clone())
    fit = fitting.SMPLify(smpl, step_size=1e-2, batch_size=B, num_iters=100, focal_length=5000., args=sargs, pose_prior=pp)
    flush.fill_(1)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pose, _, _, reproj = fit(init_pose, init_betas, init_cam, center, kp2d.clone())
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    out['c5_smplify'] = {
        'workload': f'configs[4]: DPoser prior + SMPL-X joints (joints-only LBS, 55 + 89 outputs) + 2D reprojection, 100 '
                    f'camera + 5 x 100 body Adam steps, {B} independent images on one GPU (1M images = 8 such shards)',
        'images': B, 'adam_steps': 600, 'seconds': dt, 'value': B / dt, 'unit': 'poses/s',
        'ms_per_adam_step': dt * 1e3 / 600, 'finite': bool(torch.isfinite(pose).all() and torch.isfinite(reproj).all())}
    del fit, warm, pp, smpl
    torch.cuda.empty_cache()

    # ---- SURVEY 8(f) row 3: the training step (losses.get_step_fn(train=True)): loss + hand-written backward on the
    # split-fp16 tcgen05 GEMM, clip + Adam, EMA; the reference's batch size (configs/default_amass_configs.py:22) and a large one
    from dposer_b200 import losses
    from dposer_b200.ema import ExponentialMovingAverage
    FLOP_ROW = 3 * (SCORE_FLOP_PER_ROW + 2 * (512 * 512 + 512 * 5120))     # forward + two backward products, x and time path
    tr = {}
    for tag, Bt, nst in (('reference_batch', cfg.training.batch_size, 200), ('large_batch', 16384, 30)):
        tm = synthetic.make_score_model(42).to(dev)
        tm.train()
        state = dict(optimizer=losses.get_optimizer(cfg, tm.parameters()), model=tm,
                     ema=ExponentialMovingAverage(tm.parameters(), decay=cfg.model.ema_rate), step=0)
        step_fn = losses.get_step_fn(sde, True, losses.optimization_manager(cfg), reduce_mean=cfg.training.reduce_mean,
                                     graph=True)
        toy = synthetic.toy_poses()
        host = norm.offline_normalize(toy[torch.randint(0, toy.shape[0], (Bt,))].to(dev)).cpu().pin_memory()
        data = host.to(dev)
        for _ in range(5):
            step_fn(state, data)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(nst):
            ld = step_fn(state, data)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / nst
        t0 = time.perf_counter()                      # end to end: batch from pinned host memory, loss back to the host
        for _ in range(nst):
            lv = float(step_fn(state, host.to(dev, non_blocking=True))['step_loss'])
        ms_e2e = (time.perf_counter() - t0) * 1e3 / nst
        tf = FLOP_ROW * Bt / (ms * 1e-3) / 1e12
        tr[tag] = {'batch': Bt, 'ms_per_step': ms, 'value': Bt / (ms * 1e-3), 'unit': 'poses/s', 'steps_per_s': 1e3 / ms,
                   'e2e_ms_per_step': ms_e2e, 'e2e_value': Bt / (ms_e2e * 1e-3), 'loss': lv, 'finite': bool(lv == lv and abs(lv) != float("inf")),
                   'roofline': {'bound': 'tensor', 'achieved': tf, 'peak': peaks['tc_sustained'], 'unit': 'TFLOP/s',
                                'frac': tf / peaks['tc_sustained'],
                                'note': 'algorithmic FLOP (one product); the split-fp16 GEMM executes three'}}
        del state, tm, data, host
        torch.cuda.empty_cache()
    # ---- SURVEY 8(f) row 2: bits/dim + latent code under the probability-flow ODE (likelihood.get_likelihood_fn, device RK45)
    from dposer_b200 import likelihood
    lfn = likelihood.get_likelihood_fn(sde, lambda v: v, rtol=1e-5, atol=1e-5, eps=1e-5)
    toy = synthetic.toy_poses()
    Bl = 16384
    ldata = norm.offline_normalize(toy[torch.randint(0, toy.shape[0], (Bl,))].to(dev))
    lfn(model, ldata[:64])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    bpd, _, nfe = lfn(model, ldata)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    out['f2_likelihood'] = {
        'workload': 'SURVEY 8(f)2: log-likelihood (bits/dim) and latent code of 16 384 poses, probability-flow ODE with Hutchinson '
                    'divergence, RK45 rtol = atol = 1e-5 (device-side stages / error norm, JVP contractions on tcgen05)',
        'rows': Bl, 'nfe': int(nfe), 'seconds': dt, 'value': Bl / dt, 'unit': 'poses/s', 'ms_per_function_evaluation': dt * 1e3 / nfe,
        'finite': bool(torch.isfinite(bpd).all())}
    del ldata, bpd

    # the auxiliary variant (losses.py:244-258): 10-step DDIM chain under the optimiser + SMPL-X v2v / j2j terms
    from dposer_b200.body_model import BodyModel as _BM
    Bt = cfg.training.batch_size
    tm = synthetic.make_score_model(42).to(dev)
    tm.train()
    abm = _BM(mx, num_betas=10, batch_size=Bt, model_type='smplx').to(dev)
    state = dict(optimizer=losses.get_optimizer(cfg, tm.parameters()), model=tm,
                 ema=ExponentialMovingAverage(tm.parameters(), decay=cfg.model.ema_rate), step=0)
    aux_fn = losses.get_step_fn(sde, True, losses.optimization_manager(cfg), reduce_mean=cfg.training.reduce_mean,
                                auxiliary_loss=True, denormalize=norm.offline_denormalize, body_model=abm, rot_rep='axis',
                                denoise_steps=cfg.training.denoise_steps)
    toy = synthetic.toy_poses()
    data = norm.offline_normalize(toy[torch.randint(0, toy.shape[0], (Bt,))].to(dev))
    for _ in range(3):
        aux_fn(state, data)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(20):
        ld = aux_fn(state, data)
    e1.record()
    torch.cuda.synchronize()
    ms_aux = e0.elapsed_time(e1) / 20
    tr['auxiliary'] = {'batch': Bt, 'denoise_steps': cfg.training.denoise_steps, 'ms_per_step': ms_aux, 'value': Bt / (ms_aux * 1e-3),
                       'unit': 'poses/s', 'finite': bool(torch.isfinite(ld['step_loss'])),
                       'note': 'training.auxiliary_loss = True: 10 network evaluations forward + backward, two SMPL-X LBS '
                               'forwards (10475 vertices) and one LBS backward per step'}
    del state, tm, abm, data
    torch.cuda.empty_cache()

    out['f3_train_step'] = {
        'workload': 'SURVEY 8(f)3: one training step of ScoreModelFC (sub-VP denoising score matching, per-row t, dropout 0.1, '
                    'grad clip 1.0, Adam, EMA) -- 27 tcgen05 GEMMs + elementwise kernels per step, replayed as one CUDA graph; AMASS toy poses',
        'flop_per_row_step': FLOP_ROW, **tr['reference_batch'], 'large_batch': tr['large_batch'], 'auxiliary': tr['auxiliary']}
    return out


def cpu_task_loops(budget_s=12.0):
    """configs[3] / configs[4] on the host cores: the oracle loops (pinned to the real run/motion_denoising.py and
    run/smplify.py by tests/golden/loops_golden.npz) on one sequence / four images, a few Adam steps, scaled to the
    full step count (every step costs the same)."""
    from dposer_b200 import synthetic
    from dposer_b200.body_model import JOINT_MAP_49
    from dposer_b200.misc import Posenormalizer
    from oracle import fitting_loops, fitting_ref, lbs_ref, score_ref
    torch.set_num_threads(os.cpu_count())
    sd = score_ref.make_state_dict(42)
    m = synthetic.make_body_tensors('smplx')
    norm = Posenormalizer(None, device='cpu', normalize=True, min_max=False, rot_rep='axis')
    mean, std = norm.mean_poses.cpu(), norm.std_poses.cpu()
    g = torch.Generator().manual_seed(3)
    res = {}
    Lf, steps = 60, 2
    ges, _ = synthetic.gesture_sequences()
    gt = ges[:Lf]
    _, jg = lbs_ref.body_forward(m, torch.zeros(Lf, 20), torch.cat([torch.zeros(Lf, 3), gt, torch.zeros(Lf, 99)], 1))
    noisy = jg[:, :22] + 0.04 * torch.randn(Lf, 22, 3, generator=g)
    zl = [torch.randn(Lf, 63, generator=g) for _ in range(steps)]
    t0 = time.perf_counter()
    fitting_loops.motion_denoise(sd, m, noisy, 0.01 * torch.randn(Lf, 63, generator=g), mean, std, zl, Lf, sde_N=500,
                                 iterations=1, steps_per_iter=steps, sample_trun=4.0)
    dt = (time.perf_counter() - t0) / steps
    res['c4_motion_denoise'] = {'value': Lf / (dt * 180), 'unit': 'frames/s', 'cores': os.cpu_count(), 'kind': 'port',
                                'sample': f'one 60-frame sequence, {steps} of 180 Adam steps, {dt:.2f} s per step'}
    B, iters = 4, 1
    jm = torch.tensor(JOINT_MAP_49)
    body = synthetic.toy_poses()[:B]
    glob = torch.tensor([3.14159, 0., 0.]) + 0.2 * torch.randn(B, 3, generator=g)
    cam = torch.stack([0.2 * torch.randn(B, generator=g), 0.2 * torch.randn(B, generator=g), 20 + 20 * torch.rand(B, generator=g)], 1)
    hm = m['hands_mean'][None].expand(B, -1)
    _, j = lbs_ref.body_forward(m, torch.zeros(B, 20), torch.cat([glob, body, torch.zeros(B, 9), hm], 1), cam)
    center = torch.full((B, 2), 512.)
    kp = fitting_ref.perspective_projection(j[:, jm], 5000., center)
    conf = torch.ones(B, 49)
    conf[:, 25:] = 0
    kp2d = torch.cat([kp, conf[..., None]], -1)
    zl = [torch.randn(B, 63, generator=g) for _ in range(5 * iters + 1)]
    init_pose = torch.cat([glob + 0.1, body], 1)
    t0 = time.perf_counter()
    fitting_loops.smplify(sd, m, jm, init_pose, torch.zeros(B, 10), cam + torch.tensor([0.1, -0.1, 2.0]), center, kp2d,
                          mean, std, zl, num_iters=iters, sde_N=500, hand_mean=m['hands_mean'])
    dt = (time.perf_counter() - t0) / (6 * iters)
    res['c5_smplify'] = {'value': B / (dt * 600), 'unit': 'poses/s', 'cores': os.cpu_count(), 'kind': 'port',
                         'sample': f'{B} images, {6 * iters} of 600 Adam steps, {dt:.2f} s per step'}
    # likelihood: the REAL reference's get_likelihood_fn (oracle/_ref, autograd divergence, scipy RK45) on 32 poses
    try:
        from oracle import make_ref
        mods = make_ref.import_reference()
        if mods is not None:
            ref_model_mod, ref_sde, _, _ = mods
            from lib.algorithms.advanced import likelihood as ref_lik
            cfg = synthetic.default_config()
            cfg.device = torch.device('cpu')
            torch.manual_seed(42)
            rm = ref_model_mod.ScoreModelFC(cfg, n_poses=21, pose_dim=3, hidden_dim=1024, embed_dim=512, n_blocks=2)
            rm.load_state_dict({k: v for k, v in sd.items()}, strict=False)
            rm.eval()
            lfn = ref_lik.get_likelihood_fn(ref_sde.subVPSDE(0.1, 20., N=1000), lambda v: v, rtol=1e-5, atol=1e-5, eps=1e-5)
            Bl = 32
            xl = (synthetic.toy_poses()[:Bl] - mean) / std
            t0 = time.perf_counter()
            _, _, nfe = lfn(rm, xl)
            dt = time.perf_counter() - t0
            res['f2_likelihood'] = {'value': Bl / dt, 'unit': 'poses/s', 'cores': os.cpu_count(), 'kind': 'reference',
                                    'sample': f'{Bl} poses, {nfe} function evaluations (autograd divergence, scipy RK45), {dt:.1f} s'}
    except Exception as e:                                     # the staged reference is optional
        res['f2_likelihood'] = {'error': repr(e)[:160]}
    # training step: the oracle restatement (autograd on the host cores; pinned to the real losses.get_step_fn by
    # tests/golden/train_golden.npz) at the reference's batch size
    from oracle import train_ref
    Bt, nst = 1280, 3
    osde = score_ref.SubVP(0.1, 20., 1000)
    tsd = {k: v.clone() for k, v in sd.items()}
    names = train_ref.param_names(tsd)
    opt = {k: (torch.zeros_like(tsd[k]), torch.zeros_like(tsd[k])) for k in names}
    opt['step'] = 0
    ema = {k: tsd[k].clone() for k in names}
    ema['num_updates'] = 0
    toy = synthetic.toy_poses()
    batch = (toy[torch.randint(0, toy.shape[0], (Bt,), generator=g)] - mean) / std
    times = []
    for i in range(nst + 1):
        t = torch.rand(Bt, generator=g) * (1 - 1e-5) + 1e-5
        z = torch.randn(Bt, 63, generator=g)
        masks = (torch.rand(5, Bt, 1024, generator=g) >= 0.1).to(torch.uint8)
        t0 = time.perf_counter()
        train_ref.train_step(tsd, opt, ema, osde, batch, t, z, masks, 4000 + i)
        times.append(time.perf_counter() - t0)
    dt = sum(times[1:]) / nst
    res['f3_train_step'] = {'value': Bt / dt, 'unit': 'poses/s', 'cores': os.cpu_count(), 'kind': 'port',
                            'sample': f'{nst} steps of {Bt} rows after one warm-up step, {dt * 1e3:.0f} ms per step'}
    return res


DUMP_BYTES = 63 * 10 ** 6             # array data of one --dump-outputs; with the .npy headers under 64 MB


def dump_outputs(res, out_dir, budget=DUMP_BYTES):
    """Write each array of `res` as float32 `out_dir/<name>.npy`, smallest first, each within an even share of what is
    left of `budget`.  An array larger than its share keeps a fixed sample of rows (first-dimension entries chosen by
    a seed-0 permutation, in ascending order): the same rows in every run with the same batch size."""
    os.makedirs(out_dir, exist_ok=True)
    items = sorted(res.items(), key=lambda kv: kv[1].numel())
    for i, (name, t) in enumerate(items):
        t = t.detach().float()
        share = budget // (len(items) - i)
        if t.numel() * 4 > share:
            keep = share // (t[0].numel() * 4)
            rows = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
            t = t[rows.to(t.device)]
        budget -= t.numel() * 4
        np.save(os.path.join(out_dir, f'{name}.npy'), t.cpu().numpy())


def run_gpu_arm(args):
    from dposer_b200 import _lib as L
    from dposer_b200 import dist as D
    from dposer_b200 import metric, sampling, sde_lib, steps, synthetic
    from dposer_b200.body_model import BodyModel
    from dposer_b200.misc import Posenormalizer
    import types

    rank, local, world = D.init_from_env()
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    peaks = load_peaks()
    B = default_batch(args)
    wl = args.workload
    engine = {'auto': L.ENGINE_AUTO, 'tc': L.ENGINE_TC, 'fp32': L.ENGINE_FP32}[args.engine]

    model = synthetic.make_score_model(42).to(dev)
    model.engine = engine
    cfg = synthetic.default_config()
    sde = sde_lib.subVPSDE(0.1, 20., args.sde_steps)
    norm = Posenormalizer(None, device=dev, normalize=True, min_max=False, rot_rep='axis')
    mean, std = norm.mean_poses.to(dev).float().contiguous(), norm.std_poses.to(dev).float().contiguous()
    body = synthetic.make_body_tensors('smpl')
    bm = BodyModel(body, batch_size=B, model_type='smpl').to(dev)
    fn = sampling.get_sampling_fn(cfg, sde, (B, 63), lambda x: x, 1e-3, device=dev, return_trajs=False)

    gen = torch.Generator().manual_seed(1234 + rank)
    xT_host = torch.randn(B, 63, generator=gen).pin_memory()
    lin = synthetic.lbs_inputs(B, 'smpl', seed=11 + rank)
    lbs_host = {k: v.pin_memory() for k, v in lin.items()}
    comp = None
    if wl == 'completion':
        _, mask, obs = synthetic.completion_inputs(n_partial=B // 10, hypotheses=10, seed=21 + rank)
        comp = (obs.pin_memory(), mask.pin_memory())
    task_args = types.SimpleNamespace(task='completion') if wl == 'completion' else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    pose69 = torch.zeros(B, 69, dtype=torch.float32, device=dev)     # body pose | two zero hand joints (SMPL)
    n_apd = 512                                                      # rows per rank that enter the APD (reference: 500)
    gathered = torch.empty(world * B, 63, dtype=torch.float32, device=dev) if world > 1 else None

    def to_dev(d):
        return {k: v.to(dev, non_blocking=True) for k, v in d.items()}

    def hot_path(xT, lbs_in, comp_dev):
        """inputs resident in HBM -> results resident in HBM"""
        res = {}
        if wl in ('sample_lbs', 'sample', 'completion'):
            kw = {}
            if comp_dev is not None:
                kw = dict(observation=comp_dev[0], mask=comp_dev[1], args=task_args)
            _, x0 = fn(model, z=xT, **kw)
            res['poses'] = x0
        if wl == 'sample_lbs':
            # de-normalise (run/demo.py:148) in one native kernel.  Random-init weights drive |x| to ~1e4 (SURVEY App.
            # B-1): tanh(1e-4 x) first, so that the LBS input is a plausible angle range (stated in config)
            steps.affine_cols(res['poses'], 0, 63, mean, std, pose69, inverse=True, out_ld=69, cols=63, squash=1e-4)
            out = bm(root_orient=lbs_in['root_orient'], pose_body=pose69, betas=lbs_in['betas'], trans=lbs_in['trans'])
            res['joints'], res['verts'] = out.Jtr, out.v
        elif wl == 'lbs':
            out = bm(**lbs_in)
            res['joints'], res['verts'] = out.Jtr, out.v
        return res

    results_host = {}
    apd_check = {}

    def collectives(res):
        """what the reference's evaluation does with the generated poses across ranks (run/completion.py:300-305,
        lib/utils/metric.py:8-37): gather them on every rank, APD over the gathered joints with rank-sharded rows"""
        if world == 1 or 'poses' not in res:
            return
        allp = D.all_gather_rows(res['poses'], world * B, out=gathered)
        sub = allp.view(world, B, 63)[:, :n_apd].reshape(world * n_apd, 21, 3)
        apd = metric.average_pairwise_distance(sub, group=torch.distributed.group.WORLD)
        res['apd'] = apd
        if 'ref' not in apd_check:          # once: the N-rank APD equals the 1-rank APD of the same gathered rows
            apd_check['ref'] = float(metric.average_pairwise_distance(sub))
            apd_check['sharded'] = float(apd)

    def step(e2e):
        if e2e:
            xT = xT_host.to(dev, non_blocking=True)
            lbs_in = to_dev(lbs_host)
            comp_dev = None if comp is None else tuple(c.to(dev, non_blocking=True) for c in comp)
        else:
            xT, lbs_in, comp_dev = xT_res, lbs_res, comp_res
        with torch.no_grad():
            res = hot_path(xT, lbs_in, comp_dev)
            if e2e:
                collectives(res)
        if e2e:
            for k in ('poses', 'joints', 'apd'):
                if k in res:
                    if k not in results_host:
                        results_host[k] = torch.empty(res[k].shape, dtype=res[k].dtype).pin_memory()
                    results_host[k].copy_(res[k], non_blocking=True)
        return res

    xT_res = xT_host.to(dev)
    lbs_res = to_dev(lbs_host)
    comp_res = None if comp is None else tuple(c.to(dev) for c in comp)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def timed(e2e, n_steps):
        """mean step time (ms) and the outputs of the last step"""
        total = 0.0
        for _ in range(n_steps):
            res = None                  # free the previous step's outputs first: one set alive, as in the warm-up
            flush.fill_(1)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            res = step(e2e)
            e1.record()
            torch.cuda.synchronize()
            total += D.max_over_ranks(e0.elapsed_time(e1), dev)
        return total / n_steps, res

    # the LBS stage is timed ALONE, before the sampler brings the GPU to its power cap (the roofline of a kernel
    # timed alone; inside the pipeline it runs at the capped clock and shows up in `value`)
    t_l = None
    if wl in ('sample_lbs', 'lbs'):
        with torch.no_grad():
            t_l = _ev_time(lambda: bm(**lbs_res), flush, reps=5)
    for _ in range(max(3, args.warmup)):
        step(False)
    torch.cuda.synchronize()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    ms, last = timed(False, args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(last, args.dump_outputs)
    del last
    step(True)                      # untimed: allocates the pinned result buffers the end-to-end steps copy into
    torch.cuda.synchronize()
    ms_e2e = timed(True, max(1, min(args.steps, 3)))[0]
    clk = clocks.stop() if rank == 0 else None

    # per-kernel timing of the two stages for the roofline (same stream, CUDA events, inputs resident)
    roof, roof_lbs = None, None
    with torch.no_grad():
        if wl in ('sample_lbs', 'sample', 'completion'):
            kw = {} if comp_res is None else dict(observation=comp_res[0], mask=comp_res[1], args=task_args)
            t_s = _ev_time(lambda: fn(model, z=xT_res, **kw), flush, reps=2)
            ach = SCORE_FLOP_PER_ROW * B * args.sde_steps / (t_s * 1e-3) / 1e12
            roof = {'kernel': 'tc::score_tc_kernel: fused sampler (score net x N steps)', 'bound': 'tensor', 'achieved': ach,
                    'peak': peaks['tc_sustained'], 'unit': 'TFLOP/s', 'frac': ach / peaks['tc_sustained'],
                    'traffic': SAMPLER_DRAM_BYTES_PER_ROW_STEP * B * args.sde_steps,
                    'traffic_note': 'DRAM bytes, scaled per row-step from the committed ncu capture', 'ms': t_s,
                    'peak_source': peaks['src'] + ' (bf16 sustained)'}
        if wl in ('sample_lbs', 'lbs'):
            t_l_hot = _ev_time(lambda: bm(**lbs_res), flush, reps=3)      # again, after the sampler (capped clocks)
            ach = LBS_BYTES_PER_POSE * B / (t_l * 1e-3) / 1e9
            roof_lbs = {'kernel': 'lbs_pose_kernel + lt3::lbs_fused3_kernel + lbs_gather_kernel: SMPL LBS forward',
                        'bound': 'hbm', 'achieved': ach, 'peak': peaks['hbm'],
                        'unit': 'GB/s', 'frac': ach / peaks['hbm'], 'traffic': LBS_DRAM_BYTES_PER_POSE * B,
                        'traffic_note': 'DRAM bytes, scaled per pose from the committed ncu capture (65536 poses)',
                        'algorithmic_bytes': LBS_BYTES_PER_POSE * B, 'ms': t_l, 'ms_after_sampler': t_l_hot,
                        'peak_source': peaks['src'],
                        'tensor_floor_ms': LBS_TENSOR_FLOOR_MS * B / 65536,
                        'frac_of_tensor_floor': LBS_TENSOR_FLOOR_MS * B / 65536 / t_l,
                        'tensor_floor_note': 'three fp16 products (hi.hi + hi.lo + lo.hi) for 1e-5 m: 101 tensor-pipe '
                                             'cycles per (pose, 128-vertex tile) at 1.92 GHz on 148 SMs'}
    configs = None
    if world == 1 and args.configs != 'none' and wl == 'sample_lbs':
        del bm, pose69, xT_res, lbs_res
        torch.cuda.empty_cache()
        configs = True
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    if rank != 0:
        return
    tc = engine != L.ENGINE_FP32 and B >= 64
    launches = 0
    if wl in ('sample_lbs', 'sample', 'completion'):
        launches += (1 + 1) if tc else (1 + args.sde_steps * 12)        # time table + fused / per-layer kernels
    if wl == 'sample_lbs':
        launches += 1                       # de-normalise
    if wl in ('sample_lbs', 'lbs'):
        launches += 3 if tc else 3          # pose, fused blend + skinning (or vertex), joint gather kernels
    h2d = xT_host.numel() * 4 + sum(v.numel() * 4 for v in lbs_host.values()) + \
        (0 if comp is None else sum(c.numel() * 4 for c in comp))
    d2h = sum(v.numel() * 4 for v in results_host.values())
    value = world * B / (ms * 1e-3)
    line = {'metric': 'poses/sec: DPoser reverse-SDE sampling + SMPL LBS', 'value': value, 'unit': 'poses/s',
            'n_gpus': world, 'steps': args.steps, 'warmup': max(3, args.warmup), 'ms_per_step': ms,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f16 operands / f32 accumulate (score net, tcgen05); f32 (LBS)' if tc else 'f32',
            'data': 'synthetic', 'config': workload_config(args, B), 'clocks': clk,
            'e2e': {'value': world * B / (ms_e2e * 1e-3), 'unit': 'poses/s', 'h2d_bytes_per_step': h2d,
                    'd2h_bytes_per_step': d2h, 'ms_per_step': ms_e2e,
                    'note': 'pinned host inputs -> device, hot path, generated poses + joints -> pinned host'
                            + ('; plus NCCL all-gather of the poses and the rank-sharded APD all-reduce' if world > 1 else '')},
            'gpu_launches': launches * args.steps}
    if world > 1 and apd_check:
        line['e2e']['collectives'] = {'all_gather_bytes_per_rank': B * 63 * 4, 'apd_rows': world * n_apd,
                                      'apd_sharded': apd_check['sharded'], 'apd_single_rank': apd_check['ref'],
                                      'rel_diff': abs(apd_check['sharded'] - apd_check['ref']) / max(abs(apd_check['ref']), 1e-30)}
    rf = roof if roof is not None else roof_lbs
    if roof is not None and roof_lbs is not None:
        rf = dict(roof)
        rf['lbs'] = roof_lbs
    line['roofline'] = rf
    cpu_per_row_step = None
    if not args.no_cpu and world == 1:        # the CPU arm is timed on rank 0 at N = 1 only
        line['cpu_baseline'] = cpu_reference(wl, budget_s=args.cpu_budget)
    if configs:
        if not args.no_cpu:
            try:
                t0 = time.perf_counter()
                cs = cpu_reference('sample', budget_s=6.0)
                cpu_per_row_step = 1.0 / (cs['value'] * N_SDE)
            except Exception:
                cpu_per_row_step = None
        cfgs = bench_configs(args, dev, model, peaks, flush, cpu_per_row_step)
        if roof_lbs is not None:
            cfgs['c2_lbs'] = {'workload': 'configs[1]: SMPL LBS forward only, 65536 poses', 'rows': B, 'ms': roof_lbs['ms'],
                              'value': B / (roof_lbs['ms'] * 1e-3), 'unit': 'poses/s',
                              'roofline': {k: roof_lbs[k] for k in ('bound', 'achieved', 'peak', 'unit', 'frac', 'frac_of_tensor_floor')}}
        if not args.no_cpu:
            try:
                if 'c2_lbs' in cfgs:
                    cfgs['c2_lbs']['cpu'] = cpu_reference('lbs', budget_s=5.0)
                for k, v in cpu_task_loops().items():
                    cfgs[k]['cpu'] = v
            except Exception as e:       # the CPU figures are reported baselines: never lose the GPU line over them
                cfgs['cpu_task_loops_error'] = repr(e)[:200]
        line['configs'] = cfgs
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='sample_lbs', choices=['sample_lbs', 'lbs', 'sample', 'completion'])
    ap.add_argument('--batch', type=int, default=0, help='rows per GPU (default: the BASELINE config size)')
    ap.add_argument('--sde-steps', type=int, default=N_SDE)
    ap.add_argument('--engine', default='auto', choices=['auto', 'tc', 'fp32'])
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--cpu-budget', type=float, default=20.0)
    ap.add_argument('--configs', default='all', choices=['all', 'none'], help='N=1: also measure every BASELINE config')
    ap.add_argument('--c4-sequences', type=int, default=256, help='sequences per batch of the motion-denoising config')
    ap.add_argument('--c4-batches', type=int, default=0, help='batches to time (0 = the whole config: 8192 sequences)')
    ap.add_argument('--c5-images', type=int, default=131072, help='images on this GPU for the SMPLify config')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the outputs of the last timed step (rank 0) as '
                    'float32 DIR/<name>.npy, under 64 MB in all (a fixed sample of rows where an output is larger)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs needs --impl ours (the reference arm returns no arrays)')
    if args.impl == 'reference':
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == '__main__':
    main()
