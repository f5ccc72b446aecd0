"""Host-side checks of the auxiliary training loss for rot6d (126-D) score networks: the closed-form Jacobian of the
rot6d -> axis-angle kernels (restated here in float64) against autograd, and the argument errors and refusals raised
before any library call.  No GPU needed."""
import math

import pytest
import torch

from dposer_b200 import _lib as L
from dposer_b200 import losses, sde_lib, steps, synthetic, transforms
from dposer_b200.misc import Posenormalizer


def _rotations(n, seed, lo=0.0, hi=math.pi - 1e-3):
    g = torch.Generator().manual_seed(seed)
    ax = torch.nn.functional.normalize(torch.randn(n, 3, generator=g, dtype=torch.float64), dim=1)
    th = lo + (hi - lo) * torch.rand(n, 1, generator=g, dtype=torch.float64)
    return transforms.axis_angle_to_rot6d(th * ax)


def _frame(u):
    """The kernels' frame: b1 = a1 / |a1|, b3 = (a1 x a2) / |a1 x a2|, b2 = b3 x b1; |a1|, |e|, b1 . a2."""
    a1, a2 = u[:, 0::2], u[:, 1::2]
    c = torch.linalg.cross(a1, a2)
    n1, nc = a1.norm(dim=1, keepdim=True), c.norm(dim=1, keepdim=True)
    b1, b3 = a1 / n1, c / nc
    return b1, torch.linalg.cross(b3, b1), b3, n1, nc / n1, (b1 * a2).sum(1, keepdim=True)


def _kernel_vjp(u, g):
    """fitstep.cu's closed form: gd = J_r^-T g, then the frame's derivative, columns interleaved back."""
    b1, b2, b3, n1, ne, p = _frame(u)
    phi = transforms.rot6d_to_axis_angle(u)
    th = phi.norm(dim=1, keepdim=True)
    t2 = th * th
    w, n = torch.cos(th / 2), torch.sin(th / 2)
    c = torch.where(th < 0.5, 1 / 12 + t2 * (1 / 720 + t2 / 30240), 1 / t2.clamp_min(1e-300) - w / (2 * th * n))
    gd = g - 0.5 * torch.linalg.cross(phi, g) + c * (phi * (phi * g).sum(1, keepdim=True) - t2 * g)
    ga1 = (gd[:, 2:] * b2 - gd[:, 1:2] * b3) / n1 - gd[:, :1] * p / (n1 * ne) * b3
    ga2 = gd[:, :1] * b3 / ne
    return torch.stack([ga1, ga2], dim=2).reshape(-1, 6)


def test_frame_is_gram_schmidt():
    u = torch.cat([_rotations(500, 0), torch.randn(500, 6, generator=torch.Generator().manual_seed(1),
                                                   dtype=torch.float64)])
    b1, b2, b3, *_ = _frame(u)
    assert float((torch.stack([b1, b2, b3], -1) - transforms.rot6d_to_mat3x3(u)).abs().max()) < 1e-12


def test_closed_form_vjp_matches_float64_autograd():
    """theta over [0, pi - 1e-3) with bands near 0 and pi, and unnormalised Gaussian 6-vectors."""
    gen = torch.Generator().manual_seed(2)
    u = torch.cat([_rotations(2000, 3), _rotations(300, 4, 0.0, 1e-3), _rotations(300, 5, math.pi - 0.05),
                   _rotations(300, 6, 0.45, 0.55), 3 * torch.randn(2000, 6, generator=gen, dtype=torch.float64)])
    u = u[transforms.rot6d_to_axis_angle(u).norm(dim=1) <= math.pi - 1e-3]
    g = torch.randn(u.shape[0], 3, generator=gen, dtype=torch.float64)
    leaf = u.clone().requires_grad_(True)
    (transforms.rot6d_to_axis_angle(leaf) * g).sum().backward()
    ref = leaf.grad
    err = (_kernel_vjp(u, g) - ref).abs().amax(1) / ref.abs().amax(1)
    assert float(err.max()) < 1e-8


def test_c_abi_rejects_bad_arguments():
    lib = L.load()
    p = 16    # any non-null address: the checks come before anything is read
    assert lib.dpb_rot6d_to_axis_cols(None, 126, p, p, p, 63, 4, 21, None) == L.EINVAL
    assert lib.dpb_rot6d_to_axis_cols(p, 126, None, p, p, 63, 4, 21, None) == L.EINVAL
    assert lib.dpb_rot6d_to_axis_cols(p, 125, p, p, p, 63, 4, 21, None) == L.EINVAL
    assert lib.dpb_rot6d_to_axis_cols(p, 126, p, p, p, 62, 4, 21, None) == L.EINVAL
    assert lib.dpb_rot6d_to_axis_cols(p, 126, p, p, p, 63, 4, 0, None) == L.EINVAL
    assert lib.dpb_rot6d_to_axis_cols(p, 126, p, p, p, 63, -1, 21, None) == L.EINVAL
    assert 'dpb_rot6d_to_axis_cols' in lib.dpb_last_error().decode()
    assert lib.dpb_rot6d_to_axis_cols(p, 126, p, p, p, 165, 0, 21, None) == L.OK        # nothing to do
    assert lib.dpb_rot6d_to_axis_cols_vjp(p, 126, p, p, None, 63, p, 126, 4, 21, None) == L.EINVAL
    assert lib.dpb_rot6d_to_axis_cols_vjp(p, 126, p, None, p, 63, p, 126, 4, 21, None) == L.EINVAL
    assert lib.dpb_rot6d_to_axis_cols_vjp(p, 120, p, p, p, 63, p, 126, 4, 21, None) == L.EINVAL
    assert lib.dpb_rot6d_to_axis_cols_vjp(p, 126, p, p, p, 62, p, 126, 4, 21, None) == L.EINVAL
    assert lib.dpb_rot6d_to_axis_cols_vjp(p, 126, p, p, p, 63, p, 125, 4, 21, None) == L.EINVAL
    assert lib.dpb_rot6d_to_axis_cols_vjp(p, 126, p, p, p, 63, p, 126, 4, -3, None) == L.EINVAL
    assert 'dpb_rot6d_to_axis_cols_vjp' in lib.dpb_last_error().decode()
    assert lib.dpb_rot6d_to_axis_cols_vjp(p, 126, p, p, p, 63, p, 126, 0, 21, None) == L.OK


def test_wrappers_reject_bad_arguments_before_the_library():
    f = lambda *s: torch.zeros(*s)        # noqa: E731
    x, mean, std = f(4, 130), f(126), torch.ones(126)
    with pytest.raises(RuntimeError, match='CUDA'):                     # right shapes, CPU tensors: no fallback
        steps.rot6d_to_axis_cols(x, 4, mean, std, f(4, 63))
    with pytest.raises(RuntimeError, match='CUDA'):
        steps.rot6d_to_axis_cols_vjp(x, 4, mean, std, f(4, 63), f(4, 126))
    bad_fwd = [
        (x, 4, mean, std, f(4, 62)),                # not 3 columns per joint
        (x, 4, mean, std, f(5, 63)),                # rows differ
        (x, 5, mean, std, f(4, 63)),                # the 126 columns run past the row
        (f(4, 120), 0, mean, std, f(4, 63)),
        (x, 4, f(63), std, f(4, 63)),               # statistics of the axis normaliser
        (x, 4, mean, f(120), f(4, 63)),
        (x, 4, mean, std, torch.zeros(4, 63, dtype=torch.float64)),
        (f(4, 260)[:, :130], 4, mean, std, f(4, 63)),   # non-contiguous
    ]
    for args in bad_fwd:
        with pytest.raises(ValueError):
            steps.rot6d_to_axis_cols(*args)
    bad_vjp = [
        (x, 4, mean, std, f(4, 64), f(4, 126)),
        (x, 4, mean, std, f(4, 63), f(4, 125)),
        (x, 4, mean, std, f(4, 63), f(3, 126)),
        (x, 4, f(63), std, f(4, 63), f(4, 126)),
        (x, 4, mean, f(126, 1)[:1], f(4, 63), f(4, 126)),
        (x, 10, mean, std, f(4, 63), f(4, 126)),
    ]
    for args in bad_vjp:
        with pytest.raises(ValueError):
            steps.rot6d_to_axis_cols_vjp(*args)


def _sde():
    return sde_lib.subVPSDE(0.1, 20., 1000)


def _step_fn(denormalize, rot_rep):
    cfg = synthetic.default_config()
    return losses.get_step_fn(_sde(), train=True, optimize_fn=losses.optimization_manager(cfg), auxiliary_loss=True,
                              denormalize=denormalize, body_model=object(), rot_rep=rot_rep)


def test_rot6d_auxiliary_loss_needs_a_rot6d_normaliser():
    axis = Posenormalizer(None, device='cpu', normalize=True, min_max=False, rot_rep='axis')
    for bad in (lambda v: v, axis.offline_denormalize, axis.offline_normalize,
                Posenormalizer(None, device='cpu', rot_rep='rot6d').offline_normalize):
        with pytest.raises(NotImplementedError, match="rot6d.*Posenormalizer\\(rot_rep='rot6d'\\)"):
            _step_fn(bad, 'rot6d')
    with pytest.raises(ValueError, match='rot_rep'):
        _step_fn(axis.offline_denormalize, 'quaternion')
    for normalize, min_max in ((True, True), (True, False), (False, False)):
        rot6d = Posenormalizer(None, device='cpu', normalize=normalize, min_max=min_max, rot_rep='rot6d')
        _step_fn(rot6d.offline_denormalize, 'rot6d')


def test_auxiliary_step_rejects_a_network_of_the_other_width():
    """A 63-D network under rot_rep='rot6d' is a ValueError naming both widths, before any device work."""
    rot6d = Posenormalizer(None, device='cpu', rot_rep='rot6d')
    step_fn = _step_fn(rot6d.offline_denormalize, 'rot6d')
    with pytest.raises(ValueError, match='126.*63'):
        step_fn(dict(model=synthetic.make_score_model(7), optimizer=None, ema=None, step=0), torch.zeros(4, 63))


def test_rot6d_auxiliary_loss_grad_refusals():
    m126 = synthetic.make_score_model(7, pose_dim=6)
    rot6d = Posenormalizer(None, device='cpu', rot_rep='rot6d')
    with pytest.raises(NotImplementedError, match='rot6d'):          # the CPU rule comes first
        losses.auxiliary_loss_grad(m126, _sde(), torch.zeros(4, 126), rot6d.offline_denormalize, None)
