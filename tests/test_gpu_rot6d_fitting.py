"""GPU: the native fitting chains with a rot6d (126-D) prior.  The axis -> rot6d kernels on every row against float64
autograd through transforms.axis_angle_to_rot6d, and SMPLify / MotionDenoise with a 126-D network against the oracle
loops, whose prior input is normalize(axis_angle_to_rot6d(pose)) through the torchgeometry restatement, with autograd."""
import math
import types

import pytest
import torch

from conftest import max_rel, rel_err
from dposer_b200 import _lib as L
from dposer_b200 import fitting, prior, sde_lib, steps, synthetic, transforms, utils as mutils
from dposer_b200.body_model import BodyModel, SMPLX
from dposer_b200.misc import Posenormalizer
from oracle import fitting_loops, fitting_ref as Fr, lbs_ref, tgm_ref

pytestmark = pytest.mark.gpu
D = 126
LOOP_ENGINES = [(L.ENGINE_FP32, 2e-3), (L.ENGINE_TC, 5e-3)]
SPECIAL = [0.0, 1e-8, 1e-6, 1e-4, 1e-3 - 1e-6, 1e-3 + 1e-6, 0.05, 0.1, 1.0, math.pi - 1e-4, math.pi, 2 * math.pi + 0.3]


@pytest.fixture(scope='module')
def sd126():
    from oracle import score_ref
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(score_ref, 'POSE_D', D)
        return score_ref.make_state_dict(42)


@pytest.fixture(scope='module')
def m126():
    m = synthetic.make_score_model(42, pose_dim=6).cuda()
    yield m
    m.engine = L.ENGINE_AUTO


def _norm(min_max=False, rot_rep='rot6d', device='cuda'):
    return Posenormalizer(None, device=device, normalize=True, min_max=min_max, rot_rep=rot_rep)


def _full_pose(rows, seed):
    """[rows, 165] like SMPL-X's full_pose, the 21 body joints at columns 3..65 (random axes): blocks of the 12 special
    angles alternate with blocks of 12 random angles in [0, 2 pi), so one row already holds every special angle."""
    g = torch.Generator().manual_seed(seed)
    n = rows * 21
    ax = torch.nn.functional.normalize(torch.randn(n, 3, generator=g, dtype=torch.float64), dim=1)
    th = torch.tensor(SPECIAL, dtype=torch.float64).repeat(n // len(SPECIAL) + 1)[:n]
    rnd = (torch.arange(n) // len(SPECIAL)) % 2 == 1
    th[rnd] = torch.rand(int(rnd.sum()), generator=g, dtype=torch.float64) * 2 * math.pi
    full = torch.randn(rows, 165, generator=g)
    full[:, 3:66] = (ax * th[:, None]).float().reshape(rows, 63)
    return full.cuda()


def _reference(full, std, g):
    """float64 rot6d of every joint and the VJP of g / std through it (autograd through transforms), and the VJP's own
    error bound: below theta = 1e-6 transforms takes R = I + [a]x, whose Jacobian drops B ([e_i]x K + K [e_i]x), at most
    2 theta |G| per entry (7e-4 at theta = 1e-6 where 1 / std reaches 256); zero elsewhere."""
    a = full[:, 3:66].double().reshape(-1, 3).requires_grad_(True)
    six = transforms.axis_angle_to_rot6d(a).reshape(full.shape[0], D)
    gs = g.double() / std.double()
    (gx,) = torch.autograd.grad(six, a, gs)
    th = a.detach().norm(dim=1)
    slack = torch.where(th < 1e-6, 2 * th * gs.reshape(-1, 6).abs().sum(1), torch.zeros_like(th))
    return six.detach(), gx.reshape(full.shape[0], 63), slack[:, None].expand(-1, 3).reshape(full.shape[0], 63)


def _run(full, mean, std, g):
    out = torch.full((full.shape[0], D), float('nan'), device='cuda')
    gx = torch.full((full.shape[0], 63), float('nan'), device='cuda')
    steps.axis_to_rot6d_cols(full, 3, mean, std, out)
    steps.axis_to_rot6d_cols_vjp(full, 3, std, g, gx)
    return out, gx


@pytest.mark.parametrize('rows', [1, 7, 15360, 131072])
def test_kernels_every_row_vs_float64_autograd(rows):
    full = _full_pose(rows, rows)
    g = torch.randn(rows, D, generator=torch.Generator().manual_seed(rows + 1)).cuda()
    zero, one = torch.zeros(D, device='cuda'), torch.ones(D, device='cuda')
    mean, std = (t.float().contiguous() for t in _norm().column_affine())
    assert float(std.min()) < 4e-3                        # the AMASS rot6d statistics: 1 / std amplifies x0's error
    ref, ref_gx, slack = _reference(full, std, g)
    # forward with mean 0 / std 1: <= 1e-6 absolute on every entry
    out, _ = _run(full, zero, one, g)
    assert float((out.double() - ref).abs().max()) <= 1e-6
    # with the AMASS statistics the error of x0 scales by 1 / std per column (plus the rounding of the quotient)
    out, gx = _run(full, mean, std, g)
    want = (ref - mean.double()) / std.double()
    assert bool(((out.double() - want).abs() <= 1e-6 / std.double() + 2e-7 * want.abs()).all())
    # VJP (1 / std inside): every row within 1e-5 of its own largest reference entry, beyond the reference's own error
    row = ((gx.double() - ref_gx).abs() - slack).clamp_min(0).amax(1) / ref_gx.abs().amax(1)
    assert float(row.max()) <= 1e-5, float(row.max())


def test_non_finite_joints_give_nan_in_that_joint_only():
    rows = 7
    full = _full_pose(rows, 3)
    g = torch.randn(rows, D, generator=torch.Generator().manual_seed(4)).cuda()
    mean, std = (t.float().contiguous() for t in _norm().column_affine())
    clean_out, clean_gx = _run(full, mean, std, g)
    bad = full.clone()
    hits = [(0, 0, 0, float('nan')), (2, 5, 1, float('inf')), (2, 20, 2, float('-inf')), (6, 11, 0, float('nan'))]
    for r, j, c, v in hits:
        bad[r, 3 + 3 * j + c] = v
    out, gx = _run(bad, mean, std, g)
    nan_out = torch.zeros(rows, 21, dtype=torch.bool)
    for r, j, _, _ in hits:
        nan_out[r, j] = True
    assert torch.equal(torch.isnan(out).cpu().reshape(rows, 21, 6), nan_out[..., None].expand(-1, -1, 6))
    assert torch.equal(torch.isnan(gx).cpu().reshape(rows, 21, 3), nan_out[..., None].expand(-1, -1, 3))
    keep6, keep3 = ~nan_out.repeat_interleave(6, 1).cuda(), ~nan_out.repeat_interleave(3, 1).cuda()
    assert torch.equal(out[keep6], clean_out[keep6]) and torch.equal(gx[keep3], clean_gx[keep3])


def test_wrappers_do_not_synchronise():
    full = _full_pose(512, 9)
    mean, std = (t.float().contiguous() for t in _norm().column_affine())
    out, g, gx = torch.empty(512, D, device='cuda'), torch.randn(512, D, device='cuda'), torch.empty(512, 63, device='cuda')
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        steps.axis_to_rot6d_cols(full, 3, mean, std, out)
        steps.axis_to_rot6d_cols_vjp(full, 3, std, g, gx)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert torch.isfinite(out).all() and torch.isfinite(gx).all()


def _rot6d_oracle(monkeypatch, normalizer):
    """Run the oracle loops with a rot6d prior input: their normalisation step, Fr.normalize(pose, mean, std), becomes the
    normaliser's own rule over torchgeometry's conversion, normalize(axis_angle_to_rot6d(pose)), as the reference's
    SMPLify prior computes it (run/smplify.py:109-115); autograd runs through it.  Every other oracle step is unchanged."""
    shim = types.SimpleNamespace(**{k: v for k, v in vars(Fr).items() if not k.startswith('__')})
    shim.normalize = lambda p, mean, std: normalizer.offline_normalize(
        tgm_ref.axis_angle_to_rot6d(p.reshape(-1, 3)).reshape(p.shape[0], D))
    monkeypatch.setattr(fitting_loops, 'Fr', shim)


def _smplify_problem(B, seed):
    m = synthetic.make_body_tensors('smplx')
    g = torch.Generator().manual_seed(seed)
    smpl = SMPLX(m, batch_size=B).cuda()
    jm = smpl.joint_map
    gt_body = synthetic.toy_poses()[:B]
    gt_glob = torch.tensor([3.14159, 0., 0.]) + 0.2 * torch.randn(B, 3, generator=g)
    cam = torch.stack([0.2 * torch.randn(B, generator=g), 0.2 * torch.randn(B, generator=g),
                       20 + 20 * torch.rand(B, generator=g)], 1)
    betas_gt = torch.randn(B, 10, generator=g)
    hm = m['hands_mean'][None].expand(B, -1)
    _, j = lbs_ref.body_forward(m, torch.cat([betas_gt, torch.zeros(B, 10)], 1),
                                torch.cat([gt_glob, gt_body, torch.zeros(B, 9), hm], 1), cam)
    center = torch.full((B, 2), 512.)
    kp = Fr.perspective_projection(j[:, jm], 5000., center) + 2.0 * torch.randn(B, 49, 2, generator=g)
    conf = 0.3 + 0.7 * torch.rand(B, 49, generator=g)
    conf[:, 25:] = 0.
    kp2d = torch.cat([kp, conf[..., None]], -1)
    init_pose = torch.cat([gt_glob + 0.1, smpl.mean_poses[3:66].cpu()[None].repeat(B, 1)], 1)
    init_betas = smpl.mean_shape.cpu()[None].repeat(B, 1)
    init_cam = cam + torch.tensor([0.1, -0.1, 2.0])
    return dict(m=m, smpl=smpl, jm=jm, center=center, kp2d=kp2d, init_pose=init_pose, init_betas=init_betas,
                init_cam=init_cam, g=g)


def _smplify(model, smpl, B, iters, norm, engine, p, z_list=None, graphs=False):
    args = types.SimpleNamespace(device='cuda', sde_N=500, time_strategy='3')
    model.engine = engine
    try:
        pp = prior.DPoser(batch_size=B, args=args, model=model, sde=sde_lib.subVPSDE(0.1, 20., 1000), normalizer=norm)
        fit = fitting.SMPLify(smpl, step_size=1e-2, batch_size=B, num_iters=iters, focal_length=5000., args=args,
                              pose_prior=pp)
        return fit(p['init_pose'].cuda(), p['init_betas'].cuda(), p['init_cam'].cuda(), p['center'].cuda(),
                   p['kp2d'].clone().cuda(), z_list=z_list, graphs=graphs)
    finally:
        model.engine = L.ENGINE_AUTO


@pytest.mark.parametrize('engine,tol', LOOP_ENGINES)
def test_smplify_rot6d_steps_vs_oracle(m126, sd126, engine, tol, monkeypatch):
    """2 camera + 10 body Adam steps; the update of pose, betas and camera against the oracle loop."""
    B, iters = 3, 2
    p = _smplify_problem(B, 41)
    z_list = [torch.randn(B, D, generator=p['g']) for _ in range(5 * iters + 1)]
    norm = _norm()
    _rot6d_oracle(monkeypatch, _norm(device='cpu'))
    ref_pose, ref_betas, ref_cam = fitting_loops.smplify(
        sd126, p['m'], p['jm'], p['init_pose'], p['init_betas'], p['init_cam'], p['center'], p['kp2d'].clone(), None,
        None, z_list, num_iters=iters, sde_N=500, hand_mean=p['m']['hands_mean'])
    pose, betas, cam_t, reproj = _smplify(m126, p['smpl'], B, iters, norm, engine, p, z_list=z_list)
    ip, ib, ic = p['init_pose'], p['init_betas'], p['init_cam']
    assert rel_err(pose.cpu() - ip, ref_pose - ip) < tol, rel_err(pose.cpu() - ip, ref_pose - ip)
    assert rel_err(betas.cpu() - ib, ref_betas - ib) < tol
    assert rel_err(cam_t.cpu() - ic, ref_cam - ic) < tol
    assert reproj.shape == (B, 49) and torch.isfinite(reproj).all()


def _motion_problem(rows, seed):
    m = synthetic.make_body_tensors('smplx')
    g = torch.Generator().manual_seed(seed)
    gt = synthetic.toy_poses()[:rows] + 0.02 * torch.randn(rows, 63, generator=g)
    _, j_gt = lbs_ref.body_forward(m, torch.zeros(rows, 20), torch.cat([torch.zeros(rows, 3), gt, torch.zeros(rows, 99)], 1))
    noisy = j_gt[:, :22] + 0.04 * torch.randn(rows, 22, 3, generator=g)
    init = 0.01 * torch.randn(rows, 63, generator=g)
    return m, g, gt, noisy, init


def _motion(model, m, rows, seq_len, norm):
    bm = BodyModel(m, num_betas=10, batch_size=rows, model_type='smplx').cuda()
    return fitting.MotionDenoise(synthetic.default_config(), types.SimpleNamespace(device='cuda'), model, bm,
                                 sde_lib.subVPSDE(0.1, 20., 1000), norm, sde_N=500, batch_size=rows, seq_len=seq_len)


@pytest.mark.parametrize('engine,tol,min_max', [(L.ENGINE_FP32, 2e-3, False), (L.ENGINE_TC, 5e-3, False),
                                                (L.ENGINE_FP32, 2e-3, True)])
def test_motion_denoise_rot6d_steps_vs_oracle(m126, sd126, engine, tol, min_max, monkeypatch):
    """3 Adam steps over two 6-frame sequences; min_max=True: the normaliser's min-max rule on the rot6d columns."""
    seq_len, n_seq, n_steps = 6, 2, 3
    rows = seq_len * n_seq
    m, g, gt, noisy, init = _motion_problem(rows, 31)
    z_list = [torch.randn(rows, D, generator=g) for _ in range(n_steps)]
    _rot6d_oracle(monkeypatch, _norm(min_max, device='cpu'))
    ref = fitting_loops.motion_denoise(sd126, m, noisy, init, None, None, z_list, seq_len, sde_N=500, iterations=1,
                                       steps_per_iter=n_steps, sample_trun=4.0)
    m126.engine = engine
    try:
        md = _motion(m126, m, rows, seq_len, _norm(min_max))
        md.poses = init.cuda()
        res = md.optimize(noisy.cuda(), gt_poses=gt.cuda(), time_strategy='3', sample_trun=4.0, iterations=1,
                          steps_per_iter=n_steps, z_list=z_list)
    finally:
        m126.engine = L.ENGINE_AUTO
    upd_ref, upd = ref - init, res['pose_body_raw'].cpu() - init
    assert rel_err(upd, upd_ref) < tol, rel_err(upd, upd_ref)
    assert res['MPJPE'].shape == (rows,)


def test_motion_denoise_rot6d_graphs_replay(m126):
    seq_len, n_seq = 6, 2
    rows = seq_len * n_seq
    m, _, _, noisy, init = _motion_problem(rows, 77)
    noisy, init = noisy.cuda(), init.cuda()
    kw = dict(time_strategy='3', sample_trun=4.0, iterations=1, steps_per_iter=3)

    def run(md, graphs):
        md.poses = init.clone()
        return md.optimize(noisy, graphs=graphs, **kw)['pose_body_raw']
    torch.manual_seed(5)
    plain = run(_motion(m126, m, rows, seq_len, _norm()), False)
    torch.manual_seed(5)
    md = _motion(m126, m, rows, seq_len, _norm())
    captured = run(md, True)
    replayed = run(md, True)          # same buffers, same schedule: graph replays only
    assert torch.isfinite(plain).all()
    assert rel_err(captured.cpu() - init.cpu(), plain.cpu() - init.cpu()) < 1e-5
    assert rel_err(replayed.cpu() - init.cpu(), plain.cpu() - init.cpu()) < 1e-5


def test_smplify_rot6d_graphs_match_plain_launches(m126):
    """SMPLify captures each step's graph on its first run and replays it for the rest of the call."""
    B, iters = 64, 2
    p = _smplify_problem(B, 43)
    out = []
    for graphs in (False, True):
        torch.manual_seed(9)
        out.append(_smplify(m126, p['smpl'], B, iters, _norm(), L.ENGINE_TC, p, graphs=graphs))
    ip = p['init_pose']
    assert torch.isfinite(out[0][0]).all()
    assert rel_err(out[1][0].cpu() - ip, out[0][0].cpu() - ip) < 1e-5
    assert rel_err(out[1][1].cpu(), out[0][1].cpu()) < 1e-5


def test_native_prior_gradient_matches_dposer_forward(m126):
    """One SMPLify prior gradient of the native chain (rot6d forward -> PriorStep -> VJP) against prior.DPoser.forward +
    autograd through transforms.axis_angle_to_rot6d, with the same Philox draw (slot 3, step 0)."""
    B, quan_t = 64, 700
    sde = sde_lib.subVPSDE(0.1, 20., 1000)
    norm = _norm()
    args = types.SimpleNamespace(device=torch.device('cuda'), sde_N=1000)
    pri = prior.DPoser(batch_size=B, args=args, model=m126, sde=sde, normalizer=norm)
    pose = (torch.randn(B, 69, generator=torch.Generator().manual_seed(4)) * 0.4).cuda()
    full = torch.zeros(B, 165, device='cuda')
    full[:, 3:72] = pose
    mean, std = (t.float().contiguous() for t in norm.column_affine())
    m126.engine = L.ENGINE_FP32
    try:
        p = pose.clone().requires_grad_(True)
        torch.manual_seed(1234)
        pri(p, None, quan_t).backward()
        torch.manual_seed(1234)
        seed = mutils.host_seed()
        step = steps.PriorStep(m126, sde, True, B, 'cuda')
        step.schedule([float(pri.timesteps[quan_t])])
        x0, g_axis = torch.empty(B, D, device='cuda'), torch.empty(B, 63, device='cuda')
        steps.axis_to_rot6d_cols(full, 3, mean, std, x0)
        steps.axis_to_rot6d_cols_vjp(full, 3, std, step(x0, 0, True, float(B), seed=seed, step=0), g_axis)
    finally:
        m126.engine = L.ENGINE_AUTO
    assert max_rel(g_axis, p.grad[:, :63]) < 1e-3, max_rel(g_axis, p.grad[:, :63])
