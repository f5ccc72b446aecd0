"""GPU: the Procrustes kernel (dpb_procrustes) against the float64 oracle on every row -- joint sets at SMPLify batch
size (warp layout), SMPL / SMPL-X vertices at motion-denoising and benchmark batch sizes (CTA layout), partial waves,
both sides of the layout switch, exact / mirrored / degenerate / NaN rows, point subsets, LBS output -- and its
behaviour: CUDA-graph replay, run-to-run bit identity, no host synchronisation, the Evaler keys.

Bounds: err <= 1e-5 relative or 1e-9 absolute; aligned points <= 1e-6 (input units, metres); scale (relative), R and t
<= 1e-5 where R is unique (the two smallest singular values of K differ by more than 1e-3 of the largest).  Every
output buffer starts as NaN, so a row the kernel never writes fails."""
import numpy as np
import pytest
import torch

from dposer_b200 import _lib as L
from dposer_b200 import metric, synthetic
from dposer_b200.body_model import BodyModel
from oracle import procrustes_ref as P

pytestmark = pytest.mark.gpu

WARP_ROWS_PER_CTA = 256       # rows one CTA of the warp layout owns (csrc/procrustes.cu)
WARP_MAX_POINTS = 512         # largest n_points of the warp layout
CHUNK = 4096                  # oracle rows per chunk (float64 copies of 65 536 x 6890 points would not fit)


def run(S1, S2, idx=None, aligned=True, params=True):
    """One raw dpb_procrustes launch with NaN-filled outputs."""
    B, n = S1.shape[:2]
    err = torch.full((B,), float('nan'), device='cuda')
    al = torch.full_like(S1, float('nan')) if aligned else None
    pr = torch.full((B, 13), float('nan'), device='cuda') if params else None
    ix = None if idx is None else torch.as_tensor(idx, dtype=torch.int32, device='cuda')
    L.check(L.load().dpb_procrustes(L.ptr(S1), L.ptr(S2), B, n, L.ptr(ix), 0 if ix is None else ix.numel(),
                                    L.ptr(err), L.ptr(al), L.ptr(pr), L.current_stream(S1.device)))
    return err, al, pr


def check(S1, S2, idx=None, nan_rows=(), what=''):
    """Kernel vs oracle on every row; prints the largest deviations seen and returns the kernel's outputs."""
    err, al, pr = run(S1, S2, idx)
    worst = dict(err=0.0, err_abs=0.0, aligned=0.0, params=0.0)
    nan_mask = torch.zeros(S1.shape[0], dtype=torch.bool, device='cuda')
    if len(nan_rows):
        nan_mask[torch.as_tensor(nan_rows, device='cuda')] = True
    for r0 in range(0, S1.shape[0], CHUNK):
        r1 = min(S1.shape[0], r0 + CHUNK)
        ref = P.similarity_transform(S1[r0:r1], S2[r0:r1], idx)
        bad = nan_mask[r0:r1]
        assert torch.equal(torch.isnan(ref['err']), bad), f'{what}: oracle NaN rows differ from the expected ones'
        e, re = err[r0:r1].double(), ref['err']
        assert torch.equal(torch.isnan(e), bad), f'{what}: rows {r0}+{torch.nonzero(torch.isnan(e) != bad)[:8].flatten().tolist()} NaN mismatch'
        assert torch.isnan(al[r0:r1][bad]).all() and torch.isnan(pr[r0:r1][bad]).all()
        ok = ~bad
        de = (e - re).abs()[ok]
        tol = torch.maximum(1e-5 * re.abs()[ok], torch.full_like(de, 1e-9))
        assert (de <= tol).all(), f'{what}: err off by {float(de.max()):.3e} at rows {r0}+{torch.nonzero(de > tol)[:8].flatten().tolist()}'
        da = (al[r0:r1][ok].double() - ref['aligned'][ok]).abs().amax((1, 2))
        assert (da <= 1e-6).all(), f'{what}: aligned off by {float(da.max()):.3e}'
        sv = ref['sv'][ok]
        uniq = (sv[:, 1] - sv[:, 2]) > 1e-3 * sv[:, 0]
        p = pr[r0:r1][ok].double()
        dp = torch.cat([((p[:, :1] - ref['scale'][ok, None]) / ref['scale'][ok, None].abs().clamp_min(1e-30)),
                        p[:, 1:10] - ref['R'][ok].reshape(-1, 9), p[:, 10:] - ref['t'][ok]], 1).abs().amax(1)[uniq]
        assert (dp <= 1e-5).all(), f'{what}: params off by {float(dp.max()):.3e}'
        big = re.abs()[ok] > 1e-4                                          # relative where err is not ~0
        worst = dict(err=max(worst['err'], float((de[big] / re.abs()[ok][big]).max()) if big.any() else 0.0),
                     err_abs=max(worst['err_abs'], float(de[~big].max()) if (~big).any() else 0.0),
                     aligned=max(worst['aligned'], float(da.max()) if da.numel() else 0.0),
                     params=max(worst['params'], float(dp.max()) if dp.numel() else 0.0))
        del ref
    print(f'{what}: err {worst["err"]:.2e} relative ({worst["err_abs"]:.2e} m where err < 1e-4 m), '
          f'aligned {worst["aligned"]:.2e} m, params {worst["params"]:.2e}')
    return err, al, pr


def random_rotations(B, g):
    q = torch.randn(B, 4, generator=g, device='cuda', dtype=torch.float64)
    w, x, y, z = (q / q.norm(dim=1, keepdim=True)).unbind(1)
    return torch.stack([w * w + x * x - y * y - z * z, 2 * (x * y - w * z), 2 * (x * z + w * y),
                        2 * (x * y + w * z), w * w - x * x + y * y - z * z, 2 * (y * z - w * x),
                        2 * (x * z - w * y), 2 * (y * z + w * x), w * w - x * x - y * y + z * z], 1).view(B, 3, 3)


def make_pair(B, n, seed, noise=0.02):
    """Body-sized predicted points (metres) and a noisy similarity transform of them as the target."""
    g = torch.Generator(device='cuda').manual_seed(seed)
    S1 = 0.3 * torch.randn(B, n, 3, generator=g, device='cuda') + torch.tensor([0.1, 0.9, 2.5], device='cuda')
    R = random_rotations(B, g).float()
    s = 0.8 + 0.4 * torch.rand(B, 1, 1, generator=g, device='cuda')
    t = torch.randn(B, 1, 3, generator=g, device='cuda')
    S2 = s * S1 @ R.transpose(1, 2) + t
    S2 += noise * torch.randn(S2.shape, generator=g, device='cuda')
    return S1, S2


def special_rows(S1, S2, start):
    """Overwrite rows start.. with the definition's cases; returns the rows that must be NaN."""
    g = torch.Generator(device='cuda').manual_seed(start)
    n = S1.shape[1]
    k = start
    R = random_rotations(4, g).float()
    S2[k] = 1.7 * S1[k] @ R[0].T + 0.5                                    # exact transform
    S2[k + 1] = (S1[k + 1] * torch.tensor([1.0, 1.0, -1.0], device='cuda')) @ R[1].T   # mirrored target
    S1[k + 2, :, 2] = 0.25                                                # coplanar prediction
    S2[k + 2] = 0.9 * S1[k + 2] @ R[2].T - 1.0
    S1[k + 3] = torch.linspace(-0.5, 0.5, n, device='cuda')[:, None] * torch.tensor([0.3, -0.5, 0.8], device='cuda')
    S2[k + 3] = 1.1 * S1[k + 3] @ R[3].T + 2.0                            # collinear: R not unique, err is
    S1[k + 4] = S1[k + 4, 0]                                              # coincident predicted points -> NaN
    S1[k + 5, n // 2, 1] = float('nan')
    S2[k + 6, n - 1, 0] = float('inf')
    S2[k + 7] = S2[k + 7, 3]                                              # coincident target points: scale 0
    return [k + 4, k + 5, k + 6]


@pytest.mark.parametrize('n', [49, 14])
def test_smplify_joint_sets_warp_layout(n):
    B = 131072
    S1, S2 = make_pair(B, n, n)
    nan_rows = special_rows(S1, S2, B - 8)
    err, al, pr = check(S1, S2, nan_rows=nan_rows, what=f'{B} x {n}')
    err_only, _, _ = run(S1, S2, aligned=False, params=False)
    assert torch.equal(err.nan_to_num(-1), err_only.nan_to_num(-1))
    assert float(err[B - 8]) < 1e-6 and float(err[B - 5]) < 1e-6         # exact transform, collinear
    assert float(err[B - 7]) > 0.01                                        # mirrored: the reflection is not fitted


@pytest.mark.parametrize('B,n', [(15360, 10475), (65536, 6890)])
def test_vertex_sets_cta_layout(B, n):
    S1, S2 = make_pair(B, n, B + n, noise=0.01)
    nan_rows = special_rows(S1, S2, 0)
    err, _, _ = check(S1, S2, nan_rows=nan_rows, what=f'{B} x {n}')
    err_only, _, _ = run(S1, S2, aligned=False, params=False)
    assert torch.equal(err.nan_to_num(-1), err_only.nan_to_num(-1))
    del S1, S2
    torch.cuda.empty_cache()


def test_partial_waves_and_layout_switch():
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    full = WARP_ROWS_PER_CTA * n_sm
    for B in (1, full, full + 1, 65535):
        S1, S2 = make_pair(B, 49, B)
        check(S1, S2, what=f'{B} x 49')
    for n in (WARP_MAX_POINTS, WARP_MAX_POINTS + 1):
        for B in (1, 999):
            S1, S2 = make_pair(B, n, n + B)
            nan_rows = special_rows(S1, S2, B - 8) if B > 8 else []
            check(S1, S2, nan_rows=nan_rows, what=f'{B} x {n}')


@pytest.mark.parametrize('n', [49, 6890])
def test_subset_equals_gathering_first(n):
    B = 600
    g = np.random.default_rng(n)
    idx = g.permutation(n)[:40 if n < 100 else 3000].tolist()             # any order
    outside = next(k for k in range(n) if k not in set(idx))
    S1, S2 = make_pair(B, n, 7 * n)
    S1[200, outside, 0] = float('nan')                                     # only its own aligned point
    S1[201, idx[3], 1] = float('nan')                                      # a NaN row
    err, al, pr = run(S1, S2, idx)
    ge, _, gp = run(S1[:, idx].contiguous(), S2[:, idx].contiguous())
    assert torch.nonzero(torch.isnan(err)).flatten().tolist() == [201]
    assert torch.equal(err.nan_to_num(-1), ge.nan_to_num(-1)) and torch.equal(pr.nan_to_num(-1), gp.nan_to_num(-1))
    bad = torch.isnan(al[200]).any(1)
    assert torch.nonzero(bad).flatten().tolist() == [outside]
    keep = torch.arange(B, device='cuda') != 200
    check(S1[keep], S2[keep], idx, nan_rows=[200], what=f'subset n={n}')


def test_lbs_outputs_of_synthetic_models():
    g = torch.Generator().manual_seed(11)
    for model_type, nb, B in (('smpl', 69, 512), ('smplx', 63, 256)):
        bm = BodyModel(synthetic.make_body_tensors(model_type), batch_size=B, model_type=model_type).cuda()
        pose = 0.3 * torch.randn(B, nb, generator=g)
        with torch.no_grad():
            gt = bm(pose_body=pose.cuda())
            out = bm(pose_body=(pose + 0.1 * torch.randn(B, nb, generator=g)).cuda())
        check(out.v, gt.v, what=f'{model_type} vertices')
        check(out.Jtr, gt.Jtr, what=f'{model_type} joints')


def test_graph_replay_and_run_to_run_bit_identity():
    for B, n in ((4096, 49), (300, 6890)):
        S1, S2 = make_pair(B, n, 5)
        err = torch.empty(B, device='cuda')
        al = torch.empty_like(S1)
        pr = torch.empty(B, 13, device='cuda')
        args = lambda: (L.ptr(S1), L.ptr(S2), B, n, None, 0, L.ptr(err), L.ptr(al), L.ptr(pr),  # noqa: E731
                        L.current_stream(S1.device))
        L.check(L.load().dpb_procrustes(*args()))
        eager = [x.clone() for x in (err, al, pr)]
        L.check(L.load().dpb_procrustes(*args()))
        assert all(torch.equal(a, b) for a, b in zip(eager, (err, al, pr)))
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            L.check(L.load().dpb_procrustes(*args()))
        torch.cuda.current_stream().wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            L.check(L.load().dpb_procrustes(*args()))
        for x in (err, al, pr):
            x.fill_(float('nan'))
        graph.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip(eager, (err, al, pr)))


def test_python_api_and_no_host_synchronisation():
    S1, S2 = make_pair(131072, 49, 3)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        per_row = metric.reconstruction_error(S1, S2, reduction=None)
        mean = metric.reconstruction_error(S1, S2)
        total = metric.reconstruction_error(S1, S2, reduction='sum')
    finally:
        torch.cuda.set_sync_debug_mode(0)
    err, al, pr = run(S1, S2)
    assert torch.equal(per_row, err)
    assert float(mean) == pytest.approx(float(err.double().mean()), rel=1e-7)
    assert float(total) == pytest.approx(float(err.double().sum()), rel=1e-7)
    hat, (scale, R, t) = metric.compute_similarity_transform(S1[:64], S2[:64], return_params=True)
    assert torch.equal(hat, al[:64]) and torch.equal(scale, pr[:64, 0]) and torch.equal(R.reshape(64, 9), pr[:64, 1:10])
    assert torch.equal(t, pr[:64, 10:])
    one = metric.compute_similarity_transform(S1[7], S2[7])
    assert one.shape == (49, 3) and torch.equal(one, al[7])
    assert metric.reconstruction_error(S1[7], S2[7], reduction=None).dim() == 0
    assert torch.equal(metric.reconstruction_error(S1.double(), S2.double(), reduction=None), err)


def test_evaler_procrustes_keys():
    m = synthetic.make_body_tensors('smpl')
    B, H = 64, 3
    bm = BodyModel(m, batch_size=B, model_type='smpl').cuda()
    g = torch.Generator().manual_seed(2)
    gts = (0.3 * torch.randn(B, 69, generator=g)).cuda()
    outs = gts[:, None] + (0.1 * torch.randn(B, H, 69, generator=g)).cuda()
    vert_idx = np.arange(0, 6890, 7)
    for part, vi in ((None, None), ('legs', vert_idx)):
        plain = metric.Evaler(bm, part, vi)
        pa = metric.Evaler(bm, part, vi, procrustes=True)
        r0, r1 = plain.eval_bodys(outs[:, 0], gts), pa.eval_bodys(outs[:, 0], gts)
        assert set(r0) == {'mpvpe_all', 'mpjpe_body'} and set(r1) == set(r0) | {'pa_mpvpe_all', 'pa_mpjpe_body'}
        for k in r0:
            np.testing.assert_array_equal(r0[k], r1[k])
        with torch.no_grad():
            out, gt = bm(pose_body=outs[:, 0]), bm(pose_body=gts)
        np.testing.assert_array_equal(r1['pa_mpvpe_all'],
                                      (metric.reconstruction_error(out.v, gt.v, None, pa.vert_idx) * 1000).cpu().numpy())
        np.testing.assert_array_equal(r1['pa_mpjpe_body'],
                                      (metric.reconstruction_error(out.Jtr, gt.Jtr, None, pa.joint_idx) * 1000)
                                      .cpu().numpy())
        m0, m1 = plain.multi_eval_bodys(outs, gts), pa.multi_eval_bodys(outs, gts)
        assert set(m0) == {'mpvpe_all', 'mpjpe_body'}
        for k in m0:
            np.testing.assert_array_equal(m0[k], m1[k])
        per_h = [pa.eval_bodys(outs[:, h], gts) for h in range(H)]
        for k in ('pa_mpvpe_all', 'pa_mpjpe_body'):
            np.testing.assert_array_equal(m1[k], np.min([r[k] for r in per_h], axis=0))
