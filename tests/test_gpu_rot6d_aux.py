"""GPU: the auxiliary v2v / j2j training loss of a rot6d (126-D) score network.  The rot6d -> axis-angle kernels on every
row against float64 transforms.rot6d_to_axis_angle (and float64 autograd through it), then auxiliary_loss_grad and
get_step_fn(auxiliary_loss=True, rot_rep='rot6d') against the CPU oracle (DDIM chain + LBS restatement, autograd) with the
126-D oracle weights, at the tolerances of the 63-D auxiliary tests."""
import ctypes as C
import math

import pytest
import torch

from conftest import max_rel
from dposer_b200 import _lib as L
from dposer_b200 import losses, sde_lib, steps, synthetic, transforms
from dposer_b200 import utils as mutils
from dposer_b200.body_model import BodyModel
from dposer_b200.ema import ExponentialMovingAverage
from dposer_b200.misc import Posenormalizer

pytestmark = pytest.mark.gpu
D = 126


@pytest.fixture(scope='module')
def sd126():
    from oracle import score_ref
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(score_ref, 'POSE_D', D)
        return score_ref.make_state_dict(42)


def _u(rows, seed):
    """[rows * 21, 6] float64 rot6d inputs, by joint index mod 5: valid rot6d with theta uniform in [0, pi), theta below
    1e-3, theta within 2e-3 of pi; Gaussian 6-vectors at scales 1 and 3 (what an untrained network emits)."""
    g = torch.Generator().manual_seed(seed)
    n = rows * 21
    kind = torch.arange(n) % 5
    th = torch.rand(n, generator=g, dtype=torch.float64) * math.pi
    th = torch.where(kind == 1, th * (1e-3 / math.pi), th)
    th = torch.where(kind == 2, math.pi - th * (2e-3 / math.pi), th)
    ax = torch.nn.functional.normalize(torch.randn(n, 3, generator=g, dtype=torch.float64), dim=1)
    u = transforms.axis_angle_to_rot6d(th[:, None] * ax)
    gauss = torch.randn(n, 6, generator=g, dtype=torch.float64) * torch.where(kind == 4, 3.0, 1.0)[:, None]
    return torch.where((kind >= 3)[:, None], gauss, u)


def _inputs(rows, seed, min_max, normalize):
    norm = Posenormalizer(None, device='cuda', normalize=normalize, min_max=min_max, rot_rep='rot6d')
    mean, std = (t.float().contiguous() for t in norm.column_affine())
    u = _u(rows, seed).reshape(rows, D)
    x = ((u - mean.double().cpu()) / std.double().cpu()).float()
    buf = torch.randn(rows, D + 10, generator=torch.Generator().manual_seed(seed + 1))      # x strided, from column 4
    buf[:, 4:4 + D] = x
    return buf.cuda(), mean, std


def _ref_u(buf, mean, std):
    return (buf[:, 4:4 + D].double().cpu() * std.double().cpu() + mean.double().cpu()).reshape(-1, 6)


RULES = [(False, True), (True, True), (False, False)]          # (min_max, normalize): z-score, min-max, none


@pytest.mark.parametrize('rows', [1, 127, 129, 4097, 131072])
@pytest.mark.parametrize('min_max,normalize', RULES)
def test_forward_every_row_vs_float64(rows, min_max, normalize):
    buf, mean, std = _inputs(rows, rows, min_max, normalize)
    out = torch.full((rows, 63), float('nan'), device='cuda')
    steps.rot6d_to_axis_cols(buf, 4, mean, std, out)
    # the same map written into SMPL-X full_pose's body columns 3..65 (row stride 165); the other columns stay
    full = torch.full((rows, 165), 7.0, device='cuda')
    L.check(L.load().dpb_rot6d_to_axis_cols(C.c_void_p(buf.data_ptr() + 16), buf.shape[1], L.ptr(mean), L.ptr(std),
                                            C.c_void_p(full.data_ptr() + 12), 165, rows, 21,
                                            L.current_stream(buf.device)))
    assert torch.equal(full[:, 3:66], out)
    assert bool((full[:, :3] == 7).all()) and bool((full[:, 66:] == 7).all())
    u = _ref_u(buf, mean, std)
    ref = transforms.rot6d_to_axis_angle(u)
    got = out.double().cpu().reshape(-1, 3)
    near_pi = ref.norm(dim=1) > math.pi - 1e-3              # the antipodal sign is a tie there: compare rotations
    err = (got - ref)[~near_pi].abs().max()
    assert float(err) <= 1e-6, float(err)
    if bool(near_pi.any()):
        rg, rr = (transforms.axis_angle_to_mat3x3(v[near_pi]) for v in (got, ref))
        assert float((rg - rr).abs().max()) <= 1e-6, float((rg - rr).abs().max())


@pytest.mark.parametrize('rows', [1, 127, 129, 4097, 131072])
@pytest.mark.parametrize('min_max,normalize', RULES)
def test_vjp_every_row_vs_float64_autograd(rows, min_max, normalize):
    buf, mean, std = _inputs(rows, rows + 7, min_max, normalize)
    g = torch.randn(rows, 63, generator=torch.Generator().manual_seed(rows + 8))
    gx = torch.full((rows, D), float('nan'), device='cuda')
    steps.rot6d_to_axis_cols_vjp(buf, 4, mean, std, g.cuda(), gx)
    leaf = buf[:, 4:4 + D].double().cpu().requires_grad_(True)
    u = leaf * std.double().cpu() + mean.double().cpu()
    phi = transforms.rot6d_to_axis_angle(u.reshape(-1, 6))
    (ref,) = torch.autograd.grad(phi, leaf, g.double().reshape(-1, 3))
    ok = (phi.detach().norm(dim=1) <= math.pi - 1e-3).reshape(rows, 21)
    got, ref = gx.double().cpu().reshape(rows, 21, 6), ref.reshape(rows, 21, 6)
    # relative to each row's largest entry, over the joints of the row with theta <= pi - 1e-3
    scale = torch.where(ok[..., None], ref.abs(), torch.zeros_like(ref)).amax((1, 2)).clamp_min(1e-30)
    err = torch.where(ok[..., None], (got - ref).abs(), torch.zeros_like(ref)).amax((1, 2)) / scale
    assert bool(torch.isfinite(gx).all())
    assert float(err.max()) <= 1e-5, float(err.max())


def test_degenerate_and_non_finite_joints_give_zeros():
    mean, std = torch.zeros(D, device='cuda'), torch.ones(D, device='cuda')
    x = torch.randn(8, D, generator=torch.Generator().manual_seed(3))
    six = x.view(8, 21, 6)
    six[0, 0] = 0.0                                            # a1 = a2 = 0
    six[1, 1, 0::2] = 0.0                                      # a1 = 0
    six[2, 2, 1::2] = six[2, 2, 0::2] * 2                      # a2 parallel to a1: e = 0
    six[3, 3, 1::2] = 0.0                                      # a2 = 0
    six[4, 4, 0::2] = 1e-14                                    # |a1| below the clamp
    six[5, 5, 2] = float('nan')
    six[6, 6, 3] = float('inf')
    six[7, 7, 4] = -float('inf')
    x = x.cuda()
    out = torch.full((8, 63), float('nan'), device='cuda')
    gx = torch.full((8, D), float('nan'), device='cuda')
    steps.rot6d_to_axis_cols(x, 0, mean, std, out)
    steps.rot6d_to_axis_cols_vjp(x, 0, mean, std, torch.ones(8, 63, device='cuda'), gx)
    assert bool(torch.isfinite(out).all()) and bool(torch.isfinite(gx).all())
    for r in range(8):
        assert bool((out.view(8, 21, 3)[r, r] == 0).all()) and bool((gx.view(8, 21, 6)[r, r] == 0).all()), r
    # the other joints of those rows are untouched by the rule
    ref = transforms.rot6d_to_axis_angle(x.double().cpu().view(8, 21, 6)[:, 8:].reshape(-1, 6))
    assert float((out.view(8, 21, 3)[:, 8:].double().cpu().reshape(-1, 3) - ref).abs().max()) < 1e-6


# ---------------------------------------------------------------------------------------------
# the auxiliary loss at 126-D against the oracle
# ---------------------------------------------------------------------------------------------
def _setup(B):
    model = synthetic.make_score_model(42, pose_dim=6).cuda()
    model.train()
    bm = BodyModel(synthetic.make_body_tensors('smplx'), num_betas=10, batch_size=B, model_type='smplx').cuda()
    norm = Posenormalizer(None, device='cuda', normalize=True, min_max=False, rot_rep='rot6d')
    return model, bm, norm


def _draws(B, N, seed):
    gen = torch.Generator().manual_seed(seed)
    t = torch.rand(B, generator=gen) * 0.6 + 0.2
    z = torch.randn(B, D, generator=gen)
    masks = (torch.rand(N, 5, B, 1024, generator=gen) >= 0.1).to(torch.uint8)
    return t, z, masks


def _batch(norm, B):
    toy = synthetic.toy_poses()
    return norm.offline_normalize(toy[torch.arange(B) % toy.shape[0]].cuda(), from_axis=True).cpu()


def _oracle(sd126, norm, batch, t, z, masks, N, score):
    """Losses and gradients of oracle.train_ref.aux_loss (score term included or not), with autograd."""
    from oracle import lbs_ref
    from oracle import score_ref as S
    from oracle import train_ref as T
    B = batch.shape[0]
    m = synthetic.make_body_tensors('smplx')
    mean, std = (v.cpu() for v in norm.column_affine())

    def denorm(v):
        return transforms.rot6d_to_axis_angle((v * std + mean).reshape(-1, 6)).reshape(v.shape[0], 63)

    def body_fn(pose):
        full = torch.cat([torch.zeros(B, 3), pose, torch.zeros(B, 99)], 1)
        return lbs_ref.body_forward(m, torch.zeros(B, m['shapedirs'].shape[2]), full)
    names = T.param_names(sd126)
    leaves = {k: sd126[k].clone().requires_grad_(True) for k in names}
    full = dict(sd126)
    full.update(leaves)
    loss, sl, ov, oj = T.aux_loss(full, S.SubVP(0.1, 20., 1000), batch, t, z, masks, 0.1, denorm, body_fn, N,
                                  reduce_mean=True)
    used = [k for k in names if not k.startswith('pre_dense_cond')]
    og = dict(zip(used, torch.autograd.grad(loss if score else ov + oj, [leaves[k] for k in used])))
    return {'step_loss': loss.detach(), 'score_loss': sl.detach(), 'v2v_loss': ov.detach(), 'j2j_loss': oj.detach()}, og


@pytest.mark.parametrize('B,N,tol', [(5, 3, 2e-3), (129, 3, 1.5e-2)])
def test_auxiliary_body_terms_vs_oracle(sd126, monkeypatch, B, N, tol):
    """The body-model terms alone (score term off): the chain's backward through the native rot6d -> axis-angle VJP.
    The chain's backward splits each cotangent into fp16 hi + lo parts without a scale, so entries below ~1e-3 lose bits;
    the body terms' rot6d cotangents are that small (median 8e-7 at B = 129), which leaves the gradients 8e-3 off there
    (the 63-D body terms show 3e-3 at this size).  The same run with the cotangent scaled by 2^10 on its way into the
    chain and the gradients scaled back isolates what this path adds: within 2e-4 at both sizes."""
    vjp = steps.rot6d_to_axis_cols_vjp
    t, z, masks = _draws(B, N, 12 + B)
    for scale, bound in ((1.0, tol), (1024.0, 2e-4)):
        def scaled(*args, scale=scale):
            vjp(*args)
            args[-1].mul_(scale)
        monkeypatch.setattr(steps, 'rot6d_to_axis_cols_vjp', scaled)
        model, bm, norm = _setup(B)
        batch = _batch(norm, B)
        ld = losses.auxiliary_loss_grad(model, sde_lib.subVPSDE(0.1, 20., 1000), batch.cuda(), norm.offline_denormalize,
                                        bm, denoise_steps=N, reduce_mean=True, t=t, z=z, drop_mask=masks,
                                        score_scale=0.0)
        ref, og = _oracle(sd126, norm, batch, t, z, masks, N, score=False)
        errs = {k: abs(float(ld[k]) - float(ref[k])) / float(ref[k]) for k in ('v2v_loss', 'j2j_loss')}
        assert all(v < 2e-3 for v in errs.values()), errs
        gerr = {n: max_rel(p.grad / scale, og[n].cuda()) for n, p in model.named_parameters() if n in og}
        assert max(gerr.values()) < bound, (scale, gerr)


def _state(model):
    cfg = synthetic.default_config()
    return dict(optimizer=losses.get_optimizer(cfg, model.parameters()), model=model,
                ema=ExponentialMovingAverage(model.parameters(), decay=cfg.model.ema_rate), step=4000)


def _step_fn(bm, norm, N):
    return losses.get_step_fn(sde_lib.subVPSDE(0.1, 20., 1000), train=True, optimize_fn=lambda *a, **k: None,
                              reduce_mean=True, continuous=True, auxiliary_loss=True,
                              denormalize=norm.offline_denormalize, body_model=bm, rot_rep='rot6d', denoise_steps=N)


def test_auxiliary_step_vs_oracle(sd126):
    """get_step_fn(auxiliary_loss=True, rot_rep='rot6d') with given t, z and dropout masks: the four losses, the
    gradient norm and every parameter gradient, at the tolerances of the 63-D step's test."""
    B, N = 64, 3
    model, bm, norm = _setup(B)
    t, z, masks = _draws(B, N, 5)
    batch = _batch(norm, B)
    state = _state(model)
    ld = _step_fn(bm, norm, N)(state, batch.cuda(), t=t, z=z, drop_mask=masks)
    ref, og = _oracle(sd126, norm, batch, t, z, masks, N, score=True)
    onorm = float(torch.sqrt(sum((g.double() ** 2).sum() for g in og.values())))
    errs = {k: abs(float(ld[k]) - float(ref[k])) / float(ref[k]) for k in ref}
    errs['gnorm'] = abs(state['optimizer'].grad_norm() - onorm) / onorm
    gerr = {n: max_rel(p.grad, og[n].cuda()) for n, p in model.named_parameters() if n in og}
    print('step', {k: f'{v:.2e}' for k, v in {**errs, **gerr}.items()})
    for k, tol in (('step_loss', 3e-4), ('score_loss', 3e-4), ('v2v_loss', 2e-3), ('j2j_loss', 2e-3), ('gnorm', 3e-4)):
        assert errs[k] < tol, (k, errs[k])
    assert all(v < 5e-4 for v in gerr.values()), gerr


def test_auxiliary_step_rejects_an_axis_network_under_rot6d_and_back():
    B = 4
    model, bm, norm = _setup(B)
    with pytest.raises(ValueError, match='126.*63'):
        _step_fn(bm, norm, 2)(_state(synthetic.make_score_model(42).cuda()), torch.zeros(B, 63, device='cuda'))
    axis = Posenormalizer(None, device='cuda', normalize=True, min_max=False, rot_rep='axis')
    fn = losses.get_step_fn(sde_lib.subVPSDE(0.1, 20., 1000), train=True, optimize_fn=lambda *a, **k: None,
                            auxiliary_loss=True, denormalize=axis.offline_denormalize, body_model=bm, rot_rep='axis')
    with pytest.raises(ValueError, match='63.*126'):
        fn(_state(model), torch.zeros(B, D, device='cuda'))


def test_drawn_z_is_the_philox_fill_of_the_step_seed():
    """Without z=, the step draws t from torch's generator, then a seed, then z = dpb_normal_fill_dim(seed, 0, 0, 126):
    under the same torch.manual_seed, giving that z reproduces the step bit for bit."""
    B, N = 96, 2
    model, bm, norm = _setup(B)
    masks = _draws(B, N, 9)[2]
    batch = _batch(norm, B).cuda()
    state, fn = _state(model), _step_fn(bm, norm, N)
    torch.manual_seed(1234)
    a = fn(state, batch, drop_mask=masks)
    ga = state['optimizer'].flat_g.clone()
    torch.manual_seed(1234)
    t = torch.rand(B) * (1.0 - 1e-5) + 1e-5
    seed = mutils.host_seed()
    z = torch.empty(B, D, device='cuda')
    L.check(L.load().dpb_normal_fill_dim(L.ptr(z), B, C.c_uint64(seed), C.c_uint64(0), 0, D,
                                         L.current_stream(z.device)))
    b = fn(state, batch, t=t, z=z, drop_mask=masks)
    assert all(torch.equal(a[k], b[k]) for k in a)
    assert torch.equal(ga, state['optimizer'].flat_g)
