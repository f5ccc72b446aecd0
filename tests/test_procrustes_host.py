"""Procrustes-aligned error (PA-MPJPE / PA-MPVPE) on the host: the float64 torch oracle against the per-sample numpy
SVD form, the definition's cases (exact transforms, mirrored targets, coplanar / collinear sets, NaN rows), and the
argument checks that run before any library call."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from dposer_b200 import _lib as L
from dposer_b200 import metric
from oracle import procrustes_ref as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rotation(g):
    q = g.normal(size=4)
    w, x, y, z = q / np.linalg.norm(q)
    return np.array([[w * w + x * x - y * y - z * z, 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), w * w - x * x + y * y - z * z, 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), w * w - x * x - y * y + z * z]])


def oracle_rows(S1, S2, idx=None):
    r = P.similarity_transform(torch.tensor(S1), torch.tensor(S2), idx)
    return {k: v.numpy() for k, v in r.items()}


def test_torch_oracle_equals_numpy_svd():
    g = np.random.default_rng(0)
    S1 = g.normal(size=(16, 49, 3)).astype(np.float32)
    S2 = (S1 @ rotation(g).T * 1.3 + g.normal(size=3) + 0.05 * g.normal(size=S1.shape)).astype(np.float32)
    S2[::3] = g.normal(size=S2[::3].shape)                                  # unrelated targets too
    idx = [0, 3, 7, 8, 20, 48]
    for sel in (None, idx):
        r = oracle_rows(S1, S2, sel)
        for b in range(len(S1)):
            cols = slice(None) if sel is None else sel
            h, e, s, R, t = P.similarity_transform_np(S1[b, cols], S2[b, cols])
            assert abs(r['err'][b] - e) <= 1e-12 * max(1.0, e)
            assert abs(r['scale'][b] - s) <= 1e-12
            np.testing.assert_allclose(r['R'][b], R, rtol=0, atol=1e-12)
            np.testing.assert_allclose(r['t'][b], t, rtol=0, atol=1e-12)
            np.testing.assert_allclose(r['aligned'][b, cols], h, rtol=0, atol=1e-12)
            if sel is not None:                                             # every point takes the transform
                np.testing.assert_allclose(r['aligned'][b], s * S1[b].astype(np.float64) @ R.T + t, rtol=0,
                                           atol=1e-12)


def test_exact_similarity_transforms_are_recovered():
    g = np.random.default_rng(1)
    S1 = g.normal(size=(8, 30, 3))
    Rs = np.stack([rotation(g) for _ in range(8)])
    s = g.uniform(0.3, 3.0, 8)
    t = g.normal(size=(8, 3)) * 5
    S2 = s[:, None, None] * np.einsum('bij,bkj->bki', Rs, S1) + t[:, None]
    r = oracle_rows(S1, S2)
    assert r['err'].max() < 1e-12
    np.testing.assert_allclose(r['R'], Rs, atol=1e-12)
    np.testing.assert_allclose(r['scale'], s, rtol=1e-12)
    np.testing.assert_allclose(r['t'], t, atol=1e-11)


def test_mirrored_target_gives_a_proper_rotation():
    g = np.random.default_rng(2)
    S1 = g.normal(size=(6, 40, 3)).astype(np.float32)
    S2 = (S1 * np.array([1, 1, -1]) @ rotation(g).T).astype(np.float32)      # a reflection: det(U V^T) < 0
    r = oracle_rows(S1, S2)
    for b in range(len(S1)):
        assert np.linalg.det(r['R'][b]) == pytest.approx(1.0, abs=1e-12)
        X1, X2 = S1[b] - S1[b].mean(0), S2[b] - S2[b].mean(0)
        U, _, Vh = np.linalg.svd(X1.astype(np.float64).T @ X2)
        assert np.linalg.det(U @ Vh) < 0
        assert abs(r['err'][b] - P.similarity_transform_np(S1[b], S2[b])[1]) <= 1e-12
        assert r['err'][b] > 0.1


def test_coplanar_and_collinear_rows():
    g = np.random.default_rng(3)
    plane = np.concatenate([g.normal(size=(25, 2)), np.zeros((25, 1))], 1)
    R0 = rotation(g)
    r = oracle_rows(plane[None], (2.0 * plane @ R0.T + 1.0)[None])
    assert r['err'][0] < 1e-12 and r['sv'][0, 1] - r['sv'][0, 2] > 1e-3 * r['sv'][0, 0]
    np.testing.assert_allclose(r['R'][0], R0, atol=1e-12)                 # coplanar: R is still unique
    line = np.outer(g.normal(size=20), [0.3, -0.5, 0.8])
    target = 0.7 * line @ R0.T + 2.0
    r = oracle_rows(line[None], target[None])
    assert r['err'][0] < 1e-12                                             # R is not unique, S1_hat is
    np.testing.assert_allclose(r['aligned'][0], target, atol=1e-12)
    assert r['sv'][0, 1] < 1e-12 * r['sv'][0, 0]


def test_nan_rules():
    g = np.random.default_rng(4)
    S1 = g.normal(size=(5, 10, 3)).astype(np.float32)
    S2 = g.normal(size=(5, 10, 3)).astype(np.float32)
    S1[1] = S1[1, 4]                                                       # coincident predicted points
    S1[2, 3, 1] = np.nan
    S2[3, 9, 2] = np.inf
    r = oracle_rows(S1, S2)
    for b in range(5):
        bad = b in (1, 2, 3)
        for k in ('err', 'scale', 'R', 't', 'aligned'):
            assert np.isnan(r[k][b]).all() == bad and np.isfinite(r[k][b]).all() == (not bad), (b, k)
        assert np.isnan(P.similarity_transform_np(S1[b], S2[b])[1]) == bad
    one = oracle_rows(S1[:, :1], S2[:, :1])                                # n == 1
    assert np.isnan(one['err']).all()
    sub = oracle_rows(S1, S2, [0, 1, 2])                                   # the bad points are outside the subset
    assert np.isfinite(sub['err'][[0, 2, 3, 4]]).all() and np.isnan(sub['err'][1])
    assert np.isnan(sub['aligned'][2, 3, 1]) and np.isfinite(sub['aligned'][2, :3]).all()


def test_argument_errors_before_any_library_call():
    a = torch.zeros(2, 5, 3)
    with pytest.raises(ValueError):
        metric.reconstruction_error(a, torch.zeros(2, 6, 3))                # shapes differ
    with pytest.raises(ValueError):
        metric.reconstruction_error(torch.zeros(2, 5, 2), torch.zeros(2, 5, 2))
    with pytest.raises(ValueError):
        metric.reconstruction_error(torch.zeros(2, 2, 5, 3), torch.zeros(2, 2, 5, 3))
    with pytest.raises(ValueError):
        metric.reconstruction_error(torch.zeros(0, 5, 3), torch.zeros(0, 5, 3))
    with pytest.raises(ValueError):
        metric.reconstruction_error(a.long(), a.long())                     # dtype
    with pytest.raises(ValueError):
        metric.reconstruction_error(a, a, idx=[0, 5])                       # idx out of range
    with pytest.raises(ValueError):
        metric.reconstruction_error(a, a, idx=[-1])
    with pytest.raises(ValueError):
        metric.reconstruction_error(a, a, idx=[])
    with pytest.raises(ValueError):
        metric.reconstruction_error(a, a, idx=[0.5])
    with pytest.raises(ValueError):
        metric.reconstruction_error(a, a, reduction='max')
    with pytest.raises(ValueError):
        metric.compute_similarity_transform(a, a[:1])
    with pytest.raises(RuntimeError):
        metric.reconstruction_error(a, a)                                   # no CPU fallback
    with pytest.raises(RuntimeError):
        metric.compute_similarity_transform(a[0], a[0], return_params=True)


def test_symbol_exported_declared_and_checked():
    hdr = open(os.path.join(ROOT, 'include', 'dposer_b200.h')).read()
    assert re.search(r'\bint dpb_procrustes\(', hdr)
    assert 'dpb_procrustes' in L.EXPORTS
    lib = L.load()
    buf = C.c_void_p(16)
    assert lib.dpb_procrustes(None, buf, 1, 3, None, 0, buf, None, None, None) == L.EINVAL
    assert lib.dpb_procrustes(buf, buf, 0, 3, None, 0, buf, None, None, None) == L.EINVAL
    assert lib.dpb_procrustes(buf, buf, 1, 0, None, 0, buf, None, None, None) == L.EINVAL
    assert lib.dpb_procrustes(buf, buf, 1, 3, buf, 0, buf, None, None, None) == L.EINVAL
    assert lib.dpb_procrustes(buf, buf, 1, 3, None, 0, None, None, None, None) == L.EINVAL
    assert b'dpb_procrustes' in lib.dpb_last_error()
