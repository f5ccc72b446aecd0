"""Oracle: similarity (Procrustes) alignment and the aligned point error (PA-MPJPE / PA-MPVPE).

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

**PARITY UNPINNED**: the reference's ``lib/utils/transforms.py`` is not in this tree.  The rule restated here is the
one in ``dposer_b200/metric.py``'s docstring: the similarity Procrustes with the reflection correction, as in HMR /
SPIN's ``compute_similarity_transform``.
- ``similarity_transform`` is a batched float64 restatement in torch.  It is device-generic: every tensor it builds
  lives on its input's device, so a full-size batch can be checked on the GPU.
- ``similarity_transform_np`` is the per-sample numpy form with ``numpy.linalg.svd``, the second opinion the CPU suite
  compares the torch form against.
Both centre the points after shifting by the first selected point, so that coincident points give exactly
``var1 == 0`` (NaN row) rather than round-off.
"""
import numpy as np
import torch


def similarity_transform(S1, S2, idx=None):
    """S1, S2 [B,n,3] (any float dtype, any device) -> dict of float64 tensors on that device:
    aligned [B,n,3] (every point), err [B] (mean distance over the selected points), scale [B], R [B,3,3], t [B,3],
    sv [B,3] (singular values of K, descending).  NaN rows as in the definition."""
    S1, S2 = S1.double(), S2.double()
    sel = torch.arange(S1.shape[1], device=S1.device) if idx is None else \
        torch.as_tensor(np.asarray(idx), dtype=torch.long, device=S1.device)
    P1, P2 = S1[:, sel], S2[:, sel]
    o1, o2 = P1[:, :1], P2[:, :1]
    A, Bm = P1 - o1, P2 - o2
    X1 = A - A.mean(1, keepdim=True)
    X2 = Bm - Bm.mean(1, keepdim=True)
    mu1, mu2 = o1 + A.mean(1, keepdim=True), o2 + Bm.mean(1, keepdim=True)          # [B,1,3]
    var1 = (X1 ** 2).sum((1, 2))
    finite = torch.isfinite(P1).all(2).all(1) & torch.isfinite(P2).all(2).all(1)
    bad = ~finite | (var1 == 0)
    K = X1.transpose(1, 2) @ X2                                                       # [B,3,3]
    eye = torch.eye(3, dtype=K.dtype, device=K.device).expand_as(K)
    K = torch.where(bad[:, None, None], eye, K)                                       # keep the SVD finite
    U, s, Vh = torch.linalg.svd(K)
    V = Vh.transpose(1, 2)
    Z = torch.eye(3, dtype=K.dtype, device=K.device).repeat(K.shape[0], 1, 1)
    Z[:, 2, 2] = torch.sign(torch.linalg.det(U @ V.transpose(1, 2)))
    R = V @ Z @ U.transpose(1, 2)
    scale = torch.einsum('bij,bji->b', R, K) / torch.where(bad, torch.ones_like(var1), var1)
    t = mu2[:, 0] - scale[:, None] * (R @ mu1[:, 0, :, None])[..., 0]
    aligned = scale[:, None, None] * S1 @ R.transpose(1, 2) + t[:, None]
    err = (aligned[:, sel] - P2).norm(dim=2).mean(1)
    nan = torch.tensor(float('nan'), dtype=K.dtype, device=K.device)
    return dict(aligned=torch.where(bad[:, None, None], nan, aligned), err=torch.where(bad, nan, err),
                scale=torch.where(bad, nan, scale), R=torch.where(bad[:, None, None], nan, R),
                t=torch.where(bad[:, None], nan, t), sv=s)


def similarity_transform_np(S1, S2):
    """One sample, HMR / SPIN's compute_similarity_transform in float64 numpy: S1, S2 [n,3] ->
    (S1_hat [n,3], err, scale, R, t); all NaN for a non-finite input or coincident S1 points."""
    S1, S2 = np.asarray(S1, np.float64), np.asarray(S2, np.float64)
    if not (np.isfinite(S1).all() and np.isfinite(S2).all()) or (S1 == S1[0]).all():
        return (np.full(S1.shape, np.nan), np.nan, np.nan, np.full((3, 3), np.nan), np.full(3, np.nan))
    A, Bm = S1 - S1[0], S2 - S2[0]
    mu1, mu2 = S1[0] + A.mean(0), S2[0] + Bm.mean(0)
    X1, X2 = A - A.mean(0), Bm - Bm.mean(0)
    var1 = np.sum(X1 ** 2)
    K = X1.T @ X2
    U, s, Vh = np.linalg.svd(K)
    V = Vh.T
    Z = np.eye(3)
    Z[-1, -1] *= np.sign(np.linalg.det(U @ V.T))
    R = V @ Z @ U.T
    scale = np.trace(R @ K) / var1
    t = mu2 - scale * (R @ mu1)
    S1_hat = scale * S1 @ R.T + t
    return S1_hat, np.sqrt(((S1_hat - S2) ** 2).sum(-1)).mean(), scale, R, t
