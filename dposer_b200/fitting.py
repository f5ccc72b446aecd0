"""Fitting loops of the hot path with the reference's class surface:

* ``MotionDenoise``  (run/motion_denoising.py:63-300)  Adam over the body pose with DPoser prior +
  temporal vertex smoothness + joint data term; LBS forward/backward on the native kernels.
* ``SMPLify``        (run/smplify.py:118-281)          camera stage + 5 weighted body stages.

Both accept a *batch of independent problems* (many 60-frame sequences / many images): every loss term is
normalised per problem exactly as the reference does for its single problem (SURVEY App. B-6, B-7, B-10) and
the per-problem losses are summed, so each problem sees the gradients (and Adam updates) it would see alone.

No framework op runs inside an Adam step: the computation graph of each reference loop is fixed, so the loops chain
the native kernels by hand (``steps.py``): normalise -> prior loss + closed-form gradient -> LBS forward -> loss
kernels (value + cotangents) -> LBS backward -> fused Adam.  With ``graphs=True`` every step index is captured once
into a CUDA graph and replayed for every further batch of independent problems that reuses the buffers.

The prior's input follows the score network's width, chosen once when the buffers are set up:

* 63-D (axis-angle) network: x0 = (pose - mean_poses) / std_poses, and Adam scales the prior's gradient by 1 / std.
* 126-D (rot6d) network: x0 = normalize(axis_angle_to_rot6d(pose)) with the normaliser's active rule
  (``Posenormalizer.column_affine``), and the prior's gradient returns to the axis-angle pose through the Jacobian of
  that map (``steps.axis_to_rot6d_cols`` / ``axis_to_rot6d_cols_vjp``).  This is what ``prior.DPoser.forward`` (and
  the reference's SMPLify prior, run/smplify.py:109-115) computes.  This project applies the same input to the
  motion-denoising prior: the reference's motion loop normalises without ``from_axis`` (run/motion_denoising.py:238),
  so it cannot take a rot6d network at all.

The normaliser must match the network: a rot6d network with an axis normaliser, or the reverse, raises ValueError; a
rot6d network with a normaliser that has no ``rot_rep`` (no rot6d statistics) raises NotImplementedError.
"""
import math

import numpy as np
import torch

from . import _lib as L
from . import steps as S
from . import utils as mutils
from .prior import MotionPrior

# constants.JOINT_IDS of ['OP Neck', 'OP RHip', 'OP LHip', 'Right Hip', 'Left Hip'] (run/smplify.py:136-137)
IGN_JOINTS = [1, 9, 12, 27, 28]


def _prior_input(model, normalizer, who):
    """True for a 126-D (rot6d) prior, False for a 63-D one.  A 126-D prior takes its input rule from a
    Posenormalizer(rot_rep='rot6d') (``column_affine``); a normaliser without ``rot_rep`` is read as 63-D axis
    statistics, as before, so it serves the axis prior only.  A normaliser of the other representation is a ValueError."""
    rot6d = model.pose_width == L.POSE_DIM_ROT6D
    want = 'rot6d' if rot6d else 'axis'
    rep = getattr(normalizer, 'rot_rep', None)
    if rot6d and rep is None:
        raise NotImplementedError(f'{who}: the native chain feeds a rot6d (126-D) prior through a '
                                  f"Posenormalizer(rot_rep='rot6d'); got {type(normalizer).__name__}, which has no "
                                  'rot6d statistics')
    if (rep or 'axis') != want:
        raise ValueError(f'{who}: a {model.pose_width}-D score network needs a Posenormalizer(rot_rep={want!r}), '
                         f'got rot_rep={rep!r}')
    return rot6d


def _quan_t(strategy, N, total, step, trun, sample_time, offset):
    """run/motion_denoising.py:240-247 / run/smplify.py:153-166 / run/completion.py:183-191."""
    if strategy == '1':
        return int(torch.randint(N, [1]))
    if strategy == '2':
        return int(sample_time)
    if strategy == '3':
        return N - math.floor(torch.tensor(total - step - 1) * (N / (trun * total))) - offset
    raise NotImplementedError('unsupported time sampling strategy')


class MotionDenoise(MotionPrior):
    def __init__(self, config, args, diffusion_model, body_model, sde, normalizer, sde_N=1000, dposer_weight=1.0,
                 out_path=None, debug=False, batch_size=1, seq_len=None):
        """batch_size = total rows (frames).  seq_len = frames per independent sequence (default: one sequence)."""
        self.rot6d = _prior_input(diffusion_model, normalizer, 'MotionDenoise')
        sde.N = sde_N                                            # run/motion_denoising.py:91
        super().__init__(diffusion_model, sde, config.training.continuous, batch_size)
        self.args, self.debug, self.device = args, debug, args.device
        self.body_model = body_model
        self.dposer_weight = dposer_weight
        self.out_path = out_path
        self.seq_len = seq_len or batch_size
        assert batch_size % self.seq_len == 0
        self.n_seq = batch_size // self.seq_len
        self.betas = torch.zeros((batch_size, 10), device=self.device)
        self.poses = torch.randn((batch_size, 63), device=self.device) * 0.01
        self.Normalizer = normalizer
        # per-sequence normalisation of the prior: sum / seq_len  (reference: sum / batch_size with one sequence)
        self.batch_size_divisor = self.seq_len
        self._bufs = None

    def DPoser_loss(self, x_0, vec_t, quan_t=None, weighted=False, multi_denoise=False, z=None):
        if multi_denoise:
            return self._ddim_loss(x_0, vec_t, weighted, self.batch_size_divisor, 10, z)
        return self._fused_loss(x_0, self._host_t(vec_t), bool(weighted), float(self.batch_size_divisor), z)

    def get_loss_weights(self):
        """run/motion_denoising.py:156-162."""
        return {'temp': lambda cst, it: 10. ** 1 * cst * (1 + it),
                'data': lambda cst, it: 10. ** 2 * cst / (1 + it * it),
                'dposer': lambda cst, it: 10. ** -1 * cst * (1 + it) * self.dposer_weight}

    def _buffers(self, dev):
        """Device buffers of one batch of sequences, allocated once (graph replays need stable addresses)."""
        if self._bufs is not None and self._bufs['dev'] == dev:
            return self._bufs
        core = self.body_model.core
        rows = self.batch_size
        f = lambda *s: torch.zeros(*s, dtype=torch.float32, device=dev)   # noqa: E731
        pw = self.model.pose_width
        b = dict(dev=dev, full_pose=f(rows, core.J * 3), shape=f(rows, core.S), x0=f(rows, pw), target=f(rows, 22, 3),
                 z=f(rows, pw), lbs=S.LbsStep(core, rows, dev, need_verts=True),
                 prior=S.PriorStep(self.model, self.sde, self.continuous, rows, dev), graphs=None, sched_key=None, seed=0)
        if self.rot6d:
            mean, std = self.Normalizer.column_affine()
            b['g_axis'] = f(rows, 63)                   # the prior's gradient w.r.t. the axis-angle body pose
        else:
            mean, std = self.Normalizer.mean_poses, self.Normalizer.std_poses
        b['mean'], b['std'] = mean.to(dev).float().contiguous(), std.to(dev).float().contiguous()
        b['inv_std'] = None if self.rot6d else (1.0 / b['std']).contiguous()
        b['opt'] = S.Adam(b['full_pose'], 3, 63, 0.03)
        self._bufs = b
        return b

    def optimize(self, joints3d, gt_poses=None, time_strategy='1', sample_trun=2.0, sample_time=990, iterations=5,
                 steps_per_iter=50, verbose=False, vis=False, z_list=None, graphs=False):
        """run/motion_denoising.py:199-300 (visualisation dropped) for ``n_seq`` independent sequences at once.
        ``z_list`` (parity mode): the Gaussian draw of every step; ``graphs``: CUDA-graph capture / replay of the steps
        (the draws are then Philox streams keyed by the step index, shared by later batches that replay the graphs)."""
        bm = self.body_model
        dev = joints3d.device
        L.require_cuda(joints3d, 'joints3d')
        if getattr(bm, 'model_type', 'smplx') != 'smplx':
            raise NotImplementedError('MotionDenoise runs on the SMPL-X body model, as the reference does')
        b = self._buffers(dev)
        lbs, pri = b['lbs'], b['prior']
        rows, L_, J3 = self.batch_size, self.seq_len, b['full_pose'].shape[1]
        with torch.no_grad():
            smpl_gt = bm(betas=self.betas, pose_body=gt_poses) if gt_poses is not None else None
            init_MPJPE = None
            if smpl_gt is not None:
                e = joints3d - smpl_gt.Jtr[:, :22]
                init_MPJPE = torch.mean(torch.sqrt(torch.sum(e * e, dim=2)), dim=1) * 100.
            b['target'].copy_(joints3d.detach())
            b['full_pose'].zero_()
            b['full_pose'][:, 3:66] = self.poses.detach().to(dev)          # the optimised variable lives inside full_pose
            b['shape'].zero_()
            b['shape'][:, :10] = self.betas.to(dev)
        # schedule (host, once): discrete times, loss weights
        total_steps = iterations * steps_per_iter
        timesteps = mutils.timestep_grid(self.sde, 1e-3)
        sched = []
        for it in range(iterations):
            for i in range(steps_per_iter):
                step = it * steps_per_iter + i
                qt = _quan_t(time_strategy, self.sde.N, total_steps, step, sample_trun, sample_time, 2)
                sched.append((it, float(timesteps[qt])))
        # the schedule's tables, the optimiser state and the captured step graphs live with the buffers: a further batch
        # of sequences with the same (deterministic) schedule replays the graphs of the first one
        key = None if time_strategy == '1' else (time_strategy, sample_trun, sample_time, iterations, steps_per_iter,
                                                 bool(graphs and z_list is None), self.dposer_weight)
        if key is None or b['sched_key'] != key:
            pri.schedule([t for _, t in sched])
            b['sched_key'], b['seed'] = key, (mutils.host_seed() if z_list is None else 0)
            b['graphs'] = S.StepGraphs(graphs and z_list is None)
        opt, seed, sg = b['opt'], b['seed'], b['graphs']
        opt.reset()
        wd = self.get_loss_weights()

        def one_step(k):
            it = sched[k][0]
            if self.rot6d:
                S.axis_to_rot6d_cols(b['full_pose'], 3, b['mean'], b['std'], b['x0'])
            else:
                S.affine_cols(b['full_pose'], 3, J3, b['mean'], b['std'], b['x0'])      # Posenormalizer (:238)
            z = None
            if z_list is not None:
                b['z'].copy_(z_list[k].to(dev))
                z = b['z']
            g_prior = pri(b['x0'], k, False, float(self.batch_size_divisor), z=z, seed=seed, step=k)   # DPoser_loss (:251)
            if self.rot6d:
                S.axis_to_rot6d_cols_vjp(b['full_pose'], 3, b['std'], g_prior, b['g_axis'])
                g_prior = b['g_axis']
            lbs.forward(b['shape'], b['full_pose'], None)                               # body model (:255)
            S.motion_loss(lbs, b['target'], L_, 22, wd['temp'](1.0, it), wd['data'](1.0, it))   # :256-262
            lbs.backward(b['shape'], b['full_pose'], use_verts=True)
            opt.step(lbs.g_pose, 3, J3, 1.0, g2=g_prior, off2=0, ld2=63, s2=wd['dposer'](1.0, it),
                     col_scale2=b['inv_std'])                                           # Adam (:266-268)

        for k in range(total_steps):
            sg.run(k, lambda k=k: one_step(k))
        with torch.no_grad():
            pose_final = b['full_pose'][:, 3:66].clone()
            # gaussian_smoothing(window_size=3, sigma=2) per sequence, first / last frame kept (:281-285): one native launch
            kk = torch.exp(-0.5 * ((torch.arange(3).float() - 1) / 2.0) ** 2)
            kk = kk / kk.sum()
            smooth = torch.empty_like(pose_final)
            L.check(L.load().dpb_seq_smooth3(L.ptr(pose_final), L.ptr(smooth), pose_final.shape[0], self.seq_len,
                                             pose_final.shape[1], float(kk[0]), float(kk[1]), float(kk[2]), 1,
                                             L.current_stream(pose_final.device)))
            final = bm(betas=self.betas, pose_body=smooth)
            results = {'pose_body': smooth, 'pose_body_raw': pose_final}
            if smpl_gt is not None:
                je = final.Jtr[:, :22] - smpl_gt.Jtr[:, :22]
                ve = final.v - smpl_gt.v
                results.update(init_MPJPE=init_MPJPE.cpu().numpy(),
                               MPJPE=(torch.mean(torch.sqrt(torch.sum(je * je, dim=2)), dim=1) * 100.).cpu().numpy(),
                               MPVPE=(torch.mean(torch.sqrt(torch.sum(ve * ve, dim=2)), dim=1) * 100.).cpu().numpy())
        return results


class SMPLify:
    """Single-stage SMPLify (run/smplify.py:118-281) on a batch of independent images: every image is normalised as
    the reference's batch of one (SURVEY App. B-6, B-10), the per-image losses are summed."""

    def __init__(self, body_model, step_size=1e-2, batch_size=32, num_iters=100, focal_length=5000, args=None,
                 pose_prior=None, per_problem=True):
        self.rot6d = pose_prior is not None and _prior_input(pose_prior.model, pose_prior.Normalizer, 'SMPLify')
        self.smpl = body_model
        self.device = getattr(args, 'device', None)
        self.focal_length = focal_length
        self.step_size = step_size
        self.ign_joints = IGN_JOINTS
        self.num_iters = num_iters
        self.pose_prior = pose_prior                       # a dposer_b200.prior.DPoser
        self.sde_N = args.sde_N
        self.time_strategy = args.time_strategy
        self.sample_time = round(args.sde_N * 0.9)
        self.sample_trun = 20.0
        self.loss_weights = {'pose_prior_weight': [50, 20, 10, 5, 2],
                             'shape_prior_weight': [50, 20, 10, 5, 2],
                             'angle_prior_weight': [150, 50, 30, 15, 5]}
        self.stages = len(self.loss_weights['pose_prior_weight'])
        if not per_problem:
            raise NotImplementedError('batched SMPLify solves B independent images (the reference runs B = 1)')
        self.per_problem = True
        if pose_prior is not None:
            pose_prior.batch_size = 1                       # reference runs B=1: prior = sum / 1 per image

    def sample_discrete_time(self, iteration):
        return _quan_t(self.time_strategy, self.sde_N, self.stages * self.num_iters, iteration, self.sample_trun,
                       self.sample_time, 5)

    def __call__(self, init_pose, init_betas, init_cam_t, camera_center, keypoints_2d, z_list=None, graphs=False):
        """run/smplify.py:168-281.  ``z_list`` (parity mode): the prior's Gaussian draw of every body step (+ the final
        evaluation's); ``graphs``: CUDA-graph capture / replay of the steps."""
        smpl, core = self.smpl, self.smpl.core
        dev = init_pose.device
        L.require_cuda(init_pose, 'init_pose')
        B, J3, S_ = init_pose.shape[0], core.J * 3, core.S
        lib = L.load()
        st = lambda: L.current_stream(dev)                       # noqa: E731
        f = lambda *s: torch.zeros(*s, dtype=torch.float32, device=dev)   # noqa: E731
        joints_2d = keypoints_2d[:, :, :2].contiguous().float()
        joints_conf = keypoints_2d[:, :, -1]                     # a view: the reference mutates it in place (B-13)
        center = camera_center.contiguous().float()
        focal_b, focal_s = None, 0.0
        if torch.is_tensor(self.focal_length) and self.focal_length.numel() > 1:
            focal_b = self.focal_length.to(dev).float().reshape(-1).contiguous()
        else:
            focal_s = float(self.focal_length)
        full_pose, shape, cam_t = f(B, J3), f(B, S_), init_cam_t.detach().clone().float().contiguous()
        full_pose[:, :66] = init_pose.detach()
        full_pose[:, 75:] = smpl.hand_mean.to(dev)
        shape[:, :init_betas.shape[1]] = init_betas.detach()
        init_cam = init_cam_t.detach().clone().float().contiguous()
        lbs = S.LbsStep(core, B, dev, need_verts=False)
        jmap = smpl.joint_map.to(device=dev, dtype=torch.int32).contiguous()
        K = jmap.numel()
        j49, g49, loss_b = f(B, K, 3), f(B, K, 3), f(B)
        pw = self.pose_prior.model.pose_width if self.pose_prior is not None else 63
        g_cam, g_fit_pose, g_fit_betas, x0 = f(B, 3), f(B, J3), f(B, S_), f(B, pw)
        conf = joints_conf.contiguous().float()

        def forward_joints(no_save=False):
            lbs.forward(shape, full_pose, cam_t, no_save=no_save)
            L.check(lib.dpb_joint_map_gather(L.ptr(lbs.joints), core.n_out, L.ptr(jmap), K, L.ptr(j49), B, st()))

        def backward_joints(want_transl):
            L.check(lib.dpb_joint_map_scatter(L.ptr(g49), K, L.ptr(jmap), core.n_out, L.ptr(lbs.g_joints), B, st()))
            lbs.backward(shape, full_pose, use_verts=False, want_transl=want_transl)

        # ---- stage 1: camera translation + global orientation (:208-221)
        opt_g, opt_c = S.Adam(full_pose, 0, 3, self.step_size), S.Adam(cam_t, 0, 3, self.step_size)
        sg = S.StepGraphs(graphs and z_list is None)

        def camera_step():
            forward_joints()
            L.check(lib.dpb_camera_fit_loss(L.ptr(j49), L.ptr(joints_2d), L.ptr(conf), L.ptr(center), L.ptr(cam_t),
                                            L.ptr(init_cam), L.ptr(focal_b), focal_s, 100.0, K, L.ptr(loss_b), L.ptr(g49),
                                            L.ptr(g_cam), B, st()))
            backward_joints(True)
            opt_g.step(lbs.g_pose, 0, J3)
            opt_c.step(lbs.g_transl, 0, 3, 1.0, g3=g_cam, off3=0, ld3=3, s3=1.0)

        for i in range(self.num_iters):
            sg.run(('cam', i), camera_step)
        # ---- stage 2: body pose, shape, orientation (:224-260)
        joints_conf[:, self.ign_joints] = 0.               # mutates the caller's keypoints view, as the reference
        conf = joints_conf.contiguous().float()
        pp = self.pose_prior
        total = self.stages * self.num_iters
        if pp is not None:
            pri = S.PriorStep(pp.model, pp.sde, pp.continuous, B, dev)
            qts = [self.sample_discrete_time(k) for k in range(total)] + [self.sample_discrete_time(self.num_iters - 1)]
            pri.schedule([float(pp.timesteps[int(q)]) for q in qts])
            mean, std = pp.Normalizer.column_affine() if self.rot6d else (pp.Normalizer.mean_poses,
                                                                          pp.Normalizer.std_poses)
            mean, std = mean.to(dev).float().contiguous(), std.to(dev).float().contiguous()
            inv_std = None if self.rot6d else (1.0 / std).contiguous()
            g_axis = f(B, 63) if self.rot6d else None   # the prior's gradient w.r.t. the axis-angle body pose
        opt_b, opt_s = S.Adam(full_pose, 3, 63, self.step_size), S.Adam(shape, 0, 10, self.step_size)
        opt_g2 = S.Adam(full_pose, 0, 3, self.step_size)
        seed = mutils.host_seed() if z_list is None else 0
        zbuf = f(B, pw)
        stage_weights = [dict(zip(self.loss_weights.keys(), vals)) for vals in zip(*self.loss_weights.values())]

        def body_step(k, w):
            forward_joints()
            # body_fitting_loss (fitting_losses.py:59-103): reprojection + angle + shape priors, value and cotangents
            L.check(lib.dpb_fit_loss(L.ptr(j49), L.ptr(joints_2d), L.ptr(conf), L.ptr(center), S._p(full_pose, 3), J3,
                                     L.ptr(shape), S_, K, L.ptr(focal_b), focal_s, 100.0,
                                     float(w['angle_prior_weight']), float(w['shape_prior_weight']), L.ptr(loss_b), None,
                                     L.ptr(g49), L.ptr(g_fit_pose), L.ptr(g_fit_betas), B, st()))
            backward_joints(False)
            g2 = None
            if pp is not None:
                if self.rot6d:
                    S.axis_to_rot6d_cols(full_pose, 3, mean, std, x0)         # offline_normalize(from_axis=True)
                else:
                    S.affine_cols(full_pose, 3, J3, mean, std, x0)
                z = None
                if z_list is not None:
                    zbuf.copy_(z_list[k].to(dev))
                    z = zbuf
                g2 = pri(x0, k, True, 1.0, z=z, seed=seed, step=k)          # DPoser.forward: weighted, sum / 1 per image
                if self.rot6d:
                    S.axis_to_rot6d_cols_vjp(full_pose, 3, std, g2, g_axis)
                    g2 = g_axis
            opt_b.step(lbs.g_pose, 3, J3, 1.0, g2=g2, off2=0, ld2=63, s2=float(w['pose_prior_weight']) ** 2,
                       col_scale2=inv_std if pp is not None else None, g3=g_fit_pose, off3=0, ld3=J3, s3=1.0)
            opt_s.step(lbs.g_shape, 0, S_, 1.0, g3=g_fit_betas, off3=0, ld3=S_, s3=1.0)
            opt_g2.step(lbs.g_pose, 0, J3)

        for stage, w in enumerate(stage_weights):
            for i in range(self.num_iters):
                k = stage * self.num_iters + i
                sg.run(('body', k), lambda k=k, w=w: body_step(k, w))
        # ---- final reprojection loss (:263-276)
        with torch.no_grad():
            forward_joints(no_save=True)
            reproj = f(B, K)
            L.check(lib.dpb_fit_loss(L.ptr(j49), L.ptr(joints_2d), L.ptr(conf), L.ptr(center), S._p(full_pose, 3), J3,
                                     L.ptr(shape), S_, K, L.ptr(focal_b), focal_s, 100.0, 15.2, 5.0, L.ptr(loss_b),
                                     L.ptr(reproj), None, None, None, B, st()))
        pose = full_pose[:, :66].clone()
        return pose, shape[:, :init_betas.shape[1]].clone(), cam_t, reproj
