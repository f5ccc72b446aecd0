"""Self-intersection metric (SI) on the host: the float64 oracle against brute force and hand-built cases, the test
meshes, and the argument checks that run before any library call."""
import ctypes as C

import numpy as np
import pytest
import torch

from dposer_b200 import _lib as L
from dposer_b200 import metric, synthetic
from oracle import selfisect_ref as R


@pytest.mark.parametrize('name', sorted(R.hand_cases()))
def test_hand_built_cases(name):
    P, F, expected = R.hand_cases()[name]
    sel, si = R.selection(P, F)
    if expected is None:
        assert np.isnan(si) and not sel.any()
    else:
        np.testing.assert_array_equal(sel, expected)
        assert si == 100.0 * expected.sum() / len(F)


def small_meshes():
    v, f = synthetic.uv_sphere(8, 10)
    out = [('sphere', v, f)]
    for seed, depth in [(0, 1.0), (1, 0.99), (2, 1.2), (3, 0.6)]:
        out.append((f'dent{seed}', synthetic.dented_sphere(depth, seed, 8, 10, jitter=0.05), f))
    v2, f2 = synthetic.two_spheres(6, 8)
    out.append(('two_spheres', v2, f2))
    g = np.random.default_rng(5)
    ball = g.normal(size=(len(v), 3))
    out.append(('tiny_ball', (1e-3 * ball / np.linalg.norm(ball, axis=1, keepdims=True) * g.uniform(0, 1, (len(v), 1)))
                .astype(np.float32), f))
    return out


@pytest.mark.parametrize('case', range(7))
def test_oracle_agrees_with_brute_force(case):
    name, v, f = small_meshes()[case]
    assert len(f) <= 500
    sel, si = R.selection(v, f)
    ref, si_ref = R.brute_force_selection(v, f)
    np.testing.assert_array_equal(sel, ref, err_msg=name)
    if name == 'sphere':
        assert si == 0.0


def test_test_meshes():
    v, f = synthetic.uv_sphere()
    assert v.shape == (6890, 3) and f.shape == (13776, 3)
    # closed 2-manifold: every edge in exactly two faces, opposite directions
    e = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
    assert len({tuple(x) for x in e}) == len(e)
    assert {tuple(x) for x in e} == {tuple(x) for x in e[:, ::-1]}
    assert R.selection(v, f)[1] == 0.0
    vx, fx = synthetic.uv_sphere(101, 104)
    assert len(fx) >= 20908
    assert R.selection(synthetic.dented_sphere(1.0, 3), f)[1] > 15.0
    assert R.selection(synthetic.dented_sphere(0.0, 3), f)[1] == 0.0
    assert 0.0 < R.selection(*synthetic.two_spheres())[1] < 20.0


def test_argument_errors_before_any_library_call():
    v = torch.zeros(2, 5, 3)
    f = torch.tensor([[0, 1, 2], [2, 3, 4]])
    with pytest.raises(ValueError):
        metric.self_intersections_percentage(v, torch.tensor([[0, 1, 5]]))       # id out of range
    with pytest.raises(ValueError):
        metric.self_intersections_percentage(v, torch.tensor([[0, 1, -1]]))
    with pytest.raises(ValueError):
        metric.self_intersections_percentage(v, torch.tensor([0, 1, 2]))         # faces shape
    with pytest.raises(ValueError):
        metric.self_intersections_percentage(v, f.float())                        # faces dtype
    with pytest.raises(ValueError):
        metric.self_intersections_percentage(torch.zeros(2, 5, 2), f)             # vertices shape
    with pytest.raises(ValueError):
        metric.self_intersections_percentage(torch.zeros(2, 2, 5, 3), f)
    with pytest.raises(RuntimeError):
        metric.self_intersections_percentage(v, f)                                # no CPU fallback
    with pytest.raises(RuntimeError):
        metric.self_intersections_percentage(v[0], f.numpy())


def test_c_handle_repeats_the_checks():
    lib = L.load()
    h = C.c_void_p()
    bad = np.array([[0, 1, 7]], np.int32)
    assert lib.dpb_selfisect_create(C.byref(h), bad.ctypes.data_as(C.POINTER(C.c_int32)), 1, 7, 0) == L.EINVAL
    assert b'out of range' in lib.dpb_last_error()
    big = np.zeros((32769, 3), np.int32)
    assert lib.dpb_selfisect_create(C.byref(h), big.ctypes.data_as(C.POINTER(C.c_int32)), 32769, 3, 0) == L.EUNSUPPORTED
    assert lib.dpb_selfisect_workspace_bytes(None, 4) == 0
    assert lib.dpb_selfisect_run(None, None, 1, None, None, None, 0, None) == L.EINVAL
