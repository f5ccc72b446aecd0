"""Host-side checks of the rot6d (126-D) prior in the native fitting chains: the closed-form Jacobian the two
axis -> rot6d kernels implement (restated here in float64), the conversion against the torchgeometry restatement,
Posenormalizer.column_affine, and the argument errors raised before any library call.  No GPU needed."""
import math
import types

import pytest
import torch

from dposer_b200 import _lib as L
from dposer_b200 import fitting, prior, sde_lib, steps, synthetic, transforms
from dposer_b200.misc import Posenormalizer
from oracle import tgm_ref

THETAS = [0.0, 1e-4, 1e-3, 1e-2, 0.1, 0.5, 1.0, 1.2 - 1e-7, 1.2 + 1e-7, 2.0, math.pi - 1e-4, math.pi, 4.0, 2 * math.pi,
          2 * math.pi + 0.3, 8.0, 3 * math.pi]


def _axes(n, seed):
    return torch.nn.functional.normalize(torch.randn(n, 3, generator=torch.Generator().manual_seed(seed),
                                                     dtype=torch.float64), dim=1)


def _coefs(t2, series_below=0.01):
    """A, B, C, D in float64: the Taylor series through theta^8 (the kernels' series, fitstep.cu) where
    theta^2 < series_below, else the closed forms.  The kernels switch at theta^2 = 1.44; in float64 the series'
    truncation (theta^10 / 11! for A) is visible there, so the float64 restatement switches at theta = 0.1."""
    if t2 < series_below:
        A = sum((-1) ** n * t2 ** n / math.factorial(2 * n + 1) for n in range(5))
        B = sum((-1) ** n * t2 ** n / math.factorial(2 * n + 2) for n in range(5))
        C = sum((-1) ** n * 2 * n * t2 ** (n - 1) / math.factorial(2 * n + 1) for n in range(1, 6))
        D = sum((-1) ** n * 2 * n * t2 ** (n - 1) / math.factorial(2 * n + 2) for n in range(1, 6))
        return A, B, C, D
    t = math.sqrt(t2)
    s, c = math.sin(t), math.cos(t)
    return s / t, (1 - c) / t2, (t * c - s) / t ** 3, (t * s - 2 * (1 - c)) / t ** 4


def _skew(v):
    z = torch.zeros((), dtype=v.dtype)
    return torch.stack([torch.stack([z, -v[2], v[1]]), torch.stack([v[2], z, -v[0]]), torch.stack([-v[1], v[0], z])])


def _closed_form(a):
    """rot6d(a) and its 6x3 Jacobian from R = I + A K + B K^2 and
    dR/da_i = C a_i K + A [e_i]x + D a_i K^2 + B ([e_i]x K + K [e_i]x)."""
    A, B, C, D = _coefs(float(a @ a))
    K = _skew(a)
    K2 = K @ K
    R = torch.eye(3, dtype=a.dtype) + A * K + B * K2
    J = []
    for i in range(3):
        Ei = _skew(torch.eye(3, dtype=a.dtype)[i])
        J.append((C * a[i] * K + A * Ei + D * a[i] * K2 + B * (Ei @ K + K @ Ei))[:, :2].reshape(6))
    return R[:, :2].reshape(6), torch.stack(J, 1)


def _kernel_vjp(a, g):
    """The VJP as fitstep.cu rearranges it:
    g_x = a (C <G,K> + D (a^T G a - theta^2 tr G) - 2 B tr G) + A w + B (G a + G^T a)."""
    A, B, C, D = _coefs(float(a @ a))
    G = torch.zeros(3, 3, dtype=a.dtype)
    G[:, :2] = g.reshape(3, 2)
    w = torch.stack([G[2, 1] - G[1, 2], G[0, 2] - G[2, 0], G[1, 0] - G[0, 1]])
    tr = G.trace()
    s = C * (a @ w) + D * (a @ G @ a - (a @ a) * tr) - 2 * B * tr
    return s * a + A * w + B * (G @ a + G.T @ a)


def test_closed_form_jacobian_matches_central_differences():
    """theta from 0 to 3 pi, both sides of the series threshold; h = 1e-6 keeps the differences clear of
    transforms.axis_angle_to_mat3x3's first-order branch (theta < 1e-6) except at theta = 0, where it is symmetric."""
    axes = _axes(len(THETAS), 0)
    h = 1e-6
    for th, ax in zip(THETAS, axes):
        a = th * ax
        val, J = _closed_form(a)
        assert float((val - transforms.axis_angle_to_rot6d(a[None])[0]).abs().max()) < 1e-12, th
        fd = torch.stack([(transforms.axis_angle_to_rot6d((a + h * e)[None])[0] -
                           transforms.axis_angle_to_rot6d((a - h * e)[None])[0]) / (2 * h)
                          for e in torch.eye(3, dtype=torch.float64)], 1)
        assert float((J - fd).abs().max()) < 1e-8, (th, float((J - fd).abs().max()))
        g = torch.randn(6, generator=torch.Generator().manual_seed(int(th * 100)), dtype=torch.float64)
        assert float((_kernel_vjp(a, g) - J.T @ g).abs().max()) < 1e-12, th


def test_kernel_series_within_its_bound_below_the_threshold():
    """The kernels' five-term series against the closed forms (float64) up to theta = 1.2: within 2.5e-7 relative,
    the bound fitstep.cu states for the series branch."""
    for th in torch.linspace(0.1, 1.2, 45).tolist():
        for x, y in zip(_coefs(th * th, series_below=1.44), _coefs(th * th, series_below=0.0)):
            assert abs(x - y) <= 2.5e-7 * abs(y), th


def test_axis_angle_to_rot6d_vs_torchgeometry_restatement():
    """The two differ by torchgeometry's axis a / (theta + 1e-6) and its first-order matrix for theta <= 1e-3.
    Measured gap (float64, theta in {1e-8 .. 3 pi}): values <= 1.4e-6; Jacobians <= 1.0e-3, largest at theta ~ 1e-3
    where torchgeometry switches branch, <= 1e-5 from theta = 0.1 on.  At theta = 0 exactly the restatement's autograd
    Jacobian is NaN (sqrt at 0); transforms' is [e_i]x."""
    ths = [1e-8, 1e-6, 1e-4, 9.99e-4, 1e-3, 1.001e-3, 2e-3, 1e-2, 0.05, 0.1, 0.5, 1, 2, math.pi - 1e-4, math.pi, 4,
           2 * math.pi, 2 * math.pi + 0.3, 3 * math.pi]
    a = torch.tensor(ths, dtype=torch.float64)[:, None] * _axes(len(ths), 1)
    dv = (transforms.axis_angle_to_rot6d(a) - tgm_ref.axis_angle_to_rot6d(a)).abs().amax(1)
    assert float(dv.max()) < 1.5e-6
    for th, x in zip(ths, a):
        J1 = torch.autograd.functional.jacobian(transforms.axis_angle_to_rot6d, x[None]).reshape(6, 3)
        J2 = torch.autograd.functional.jacobian(tgm_ref.axis_angle_to_rot6d, x[None]).reshape(6, 3)
        gap = float((J1 - J2).abs().max())
        assert gap < (1.2e-3 if th < 0.1 else 1.2e-5), (th, gap)
    J0 = torch.autograd.functional.jacobian(transforms.axis_angle_to_rot6d, torch.zeros(1, 3, dtype=torch.float64))
    eye = torch.eye(3, dtype=torch.float64)
    assert torch.equal(J0.reshape(6, 3), torch.stack([_skew(e)[:, :2].reshape(6) for e in eye], 1))


@pytest.mark.parametrize('rot_rep', ['axis', 'rot6d'])
@pytest.mark.parametrize('normalize,min_max', [(True, True), (True, False), (False, False)])
def test_column_affine_matches_offline_normalize(rot_rep, normalize, min_max):
    norm = Posenormalizer(None, device='cpu', normalize=normalize, min_max=min_max, rot_rep=rot_rep)
    mean, std = norm.column_affine()
    D = 63 if rot_rep == 'axis' else 126
    assert mean.shape == (D,) and std.shape == (D,)
    x = torch.randn(40, D, generator=torch.Generator().manual_seed(3)) * 0.5
    ref = norm.offline_normalize(x)
    assert float(((x - mean) / std - ref).abs().max()) <= 1e-5 * float(ref.abs().max())
    if rot_rep == 'rot6d':       # from_axis: the conversion first, as the native chains do
        aa = torch.randn(40, 63, generator=torch.Generator().manual_seed(4)) * 0.5
        six = transforms.axis_angle_to_rot6d(aa.reshape(-1, 3)).reshape(40, 126)
        ref = norm.offline_normalize(aa, from_axis=True)
        assert float(((six - mean) / std - ref).abs().max()) <= 1e-5 * float(ref.abs().max())


def test_wrappers_reject_bad_arguments_before_the_library():
    f = lambda *s: torch.zeros(*s)        # noqa: E731
    full, mean, std = f(4, 165), f(126), torch.ones(126)
    with pytest.raises(RuntimeError, match='CUDA'):                     # right shapes, CPU tensors: no fallback
        steps.axis_to_rot6d_cols(full, 3, mean, std, f(4, 126))
    with pytest.raises(RuntimeError, match='CUDA'):
        steps.axis_to_rot6d_cols_vjp(full, 3, std, f(4, 126), f(4, 63))
    bad_fwd = [
        (full, 3, mean, std, f(4, 125)),            # not 6 columns per joint
        (full, 3, mean, std, f(5, 126)),            # rows differ
        (full, 160, mean, std, f(4, 126)),          # the 63 columns run past the row
        (f(4, 60), 0, mean, std, f(4, 126)),
        (full, 3, f(63), std, f(4, 126)),           # statistics of the axis normaliser
        (full, 3, mean, f(120), f(4, 126)),
        (full, 3, mean, std, torch.zeros(4, 126, dtype=torch.float64)),
        (full[:, :100], 3, mean, std, f(4, 126)),   # non-contiguous
    ]
    for args in bad_fwd:
        with pytest.raises(ValueError):
            steps.axis_to_rot6d_cols(*args)
    bad_vjp = [
        (full, 3, std, f(4, 126), f(4, 64)),
        (full, 3, std, f(4, 126), f(3, 63)),
        (full, 3, std, f(4, 120), f(4, 63)),
        (full, 3, f(63), f(4, 126), f(4, 63)),
        (full, 130, std, f(4, 126), f(4, 63)),
    ]
    for args in bad_vjp:
        with pytest.raises(ValueError):
            steps.axis_to_rot6d_cols_vjp(*args)


def test_c_abi_rejects_bad_arguments():
    lib = L.load()
    p = 16    # any non-null address: the checks come before anything is read
    assert lib.dpb_axis_to_rot6d_cols(None, 165, p, p, p, 126, 4, 21, None) == L.EINVAL
    assert lib.dpb_axis_to_rot6d_cols(p, 62, p, p, p, 126, 4, 21, None) == L.EINVAL
    assert lib.dpb_axis_to_rot6d_cols(p, 165, p, p, p, 125, 4, 21, None) == L.EINVAL
    assert lib.dpb_axis_to_rot6d_cols(p, 165, p, p, p, 126, 4, 0, None) == L.EINVAL
    assert lib.dpb_axis_to_rot6d_cols(p, 165, p, p, p, 126, -1, 21, None) == L.EINVAL
    assert 'dpb_axis_to_rot6d_cols' in lib.dpb_last_error().decode()
    assert lib.dpb_axis_to_rot6d_cols(p, 165, p, p, p, 126, 0, 21, None) == L.OK        # nothing to do
    assert lib.dpb_axis_to_rot6d_cols_vjp(p, 165, None, p, 126, p, 63, 4, 21, None) == L.EINVAL
    assert lib.dpb_axis_to_rot6d_cols_vjp(p, 165, p, p, 120, p, 63, 4, 21, None) == L.EINVAL
    assert lib.dpb_axis_to_rot6d_cols_vjp(p, 165, p, p, 126, p, 62, 4, 21, None) == L.EINVAL
    assert lib.dpb_axis_to_rot6d_cols_vjp(p, 165, p, p, 126, p, 63, 0, 21, None) == L.OK


def _md(model, normalizer):
    args = types.SimpleNamespace(device=torch.device('cpu'))
    return fitting.MotionDenoise(synthetic.default_config(), args, model, None, sde_lib.subVPSDE(0.1, 20., 1000),
                                 normalizer, batch_size=4)


def _smplify(model, normalizer):
    args = types.SimpleNamespace(device=torch.device('cpu'), sde_N=500, time_strategy='3')
    pp = prior.DPoser(batch_size=1, args=args, model=model, sde=sde_lib.subVPSDE(0.1, 20., 1000), normalizer=normalizer)
    return fitting.SMPLify(None, batch_size=1, args=args, pose_prior=pp)


@pytest.fixture(scope='module')
def models():
    return synthetic.make_score_model(7), synthetic.make_score_model(7, pose_dim=6)


def test_fitting_loops_take_a_rot6d_prior(models):
    _, m126 = models
    rot6d = Posenormalizer(None, device='cpu', normalize=True, min_max=False, rot_rep='rot6d')
    assert _md(m126, rot6d).rot6d and _smplify(m126, rot6d).rot6d


@pytest.mark.parametrize('build', [_md, _smplify])
def test_fitting_loops_reject_a_normaliser_of_the_other_representation(models, build):
    m63, m126 = models
    axis = Posenormalizer(None, device='cpu', normalize=True, min_max=False, rot_rep='axis')
    rot6d = Posenormalizer(None, device='cpu', normalize=True, min_max=False, rot_rep='rot6d')
    with pytest.raises(ValueError, match="rot_rep='rot6d'"):
        build(m126, axis)
    with pytest.raises(NotImplementedError, match='rot6d'):     # no rot_rep: axis statistics at most
        build(m126, object())
    with pytest.raises(ValueError, match="rot_rep='axis'"):
        build(m63, rot6d)
    assert not build(m63, axis).rot6d
