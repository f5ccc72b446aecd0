"""GPU: the self-intersection kernel's per-face selection equals the float64 oracle's exactly (hand-built cases,
deformed SMPL- and SMPL-X-size spheres, two overlapping spheres, a degenerate mesh, LBS output), at batch scale, under
CUDA-graph capture, bit-identically across runs."""
import numpy as np
import pytest
import torch

from dposer_b200 import metric, synthetic
from dposer_b200.body_model import BodyModel
from oracle import selfisect_ref as R

pytestmark = pytest.mark.gpu

N_SMPL, N_SMPLX = 48, 16


def depths(n, seed):
    """SI from 0 to about 20 %: undeformed, dents that stay inside, mirrored caps (depth 1) and caps pushed through."""
    g = np.random.default_rng(seed)
    return np.concatenate([[0.0, 0.5, 0.9], np.ones(n // 4), 1 + 0.02 * g.uniform(-1, 1, n // 4),
                           g.uniform(0.95, 1.5, n - 3 - 2 * (n // 4))])


def assert_same(sel, ref, v, f, what):
    sel, ref = np.asarray(sel, bool), np.asarray(ref, bool)
    if (sel == ref).all():
        return
    bad = np.nonzero(sel != ref)[0]
    lines = [f'{what}: {len(bad)} faces differ (kernel / oracle selected {sel.sum()} / {ref.sum()})']
    for face in bad[:5]:
        lines.append(f'  face {face}: kernel {sel[face]}, oracle {ref[face]}; partners (g, s, oracle hit, '
                     f'min |n.(x-q0)|): {[r for r in R.explain(v, f, face) if r[2] or r[3] < 1e-6][:6]}')
    raise AssertionError('\n'.join(lines))


@pytest.fixture(scope='module')
def smpl_set():
    _, f = synthetic.uv_sphere()
    vs = np.stack([synthetic.dented_sphere(d, 100 + r) for r, d in enumerate(depths(N_SMPL, 1))])
    refs = [R.selection(v, f) for v in vs]
    return vs, f, np.stack([r[0] for r in refs]), np.array([r[1] for r in refs])


def run(v, f, **kw):
    return metric.self_intersections_percentage(torch.as_tensor(v).cuda(), torch.as_tensor(f), **kw)


def test_hand_built_cases():
    for name, (P, F, expected) in R.hand_cases().items():
        si, sel = run(P, F, return_selection=True)
        assert si.dtype == torch.float32 and si.dim() == 0
        if expected is None:
            assert torch.isnan(si) and not sel.any(), name
        else:
            assert_same(sel.cpu().numpy(), expected, P, F, name)
            assert float(si) == np.float32(100.0 * expected.sum() / len(F)), name


def test_deformed_smpl_size_meshes(smpl_set):
    vs, f, ref, ref_si = smpl_set
    assert ref_si.min() == 0.0 and ref_si.max() > 15.0
    si, sel = run(vs, f, return_selection=True)
    for r in range(len(vs)):
        assert_same(sel[r].cpu().numpy(), ref[r], vs[r], f, f'row {r}')
    np.testing.assert_array_equal(si.cpu().numpy(), ref_si.astype(np.float32))


def test_smplx_size_meshes():
    _, f = synthetic.uv_sphere(101, 104)
    assert len(f) >= 20908
    vs = np.stack([synthetic.dented_sphere(d, 200 + r, 101, 104) for r, d in enumerate(depths(N_SMPLX, 2))])
    si, sel = run(vs, f, return_selection=True)
    for r in range(len(vs)):
        assert_same(sel[r].cpu().numpy(), R.selection(vs[r], f)[0], vs[r], f, f'smplx row {r}')


def test_two_spheres_and_degenerate_mesh():
    v, f = synthetic.two_spheres()
    si, sel = run(v, f, return_selection=True)
    ref, ref_si = R.selection(v, f)
    assert_same(sel.cpu().numpy(), ref, v, f, 'two spheres')
    assert float(si) == np.float32(ref_si) and ref_si > 0
    # every vertex in a ball of radius 1e-3: every face in one cell, quadratic work
    _, f = synthetic.uv_sphere(10, 12)
    g = np.random.default_rng(3)
    v = (1e-3 * g.uniform(-1, 1, (2 + 10 * 12, 3))).astype(np.float32)
    si, sel = run(v, f, return_selection=True)
    assert_same(sel.cpu().numpy(), R.selection(v, f)[0], v, f, 'tiny ball')
    # a collapsed mesh (every vertex at one point: every face has zero area)
    si, sel = run(np.zeros_like(v), f, return_selection=True)
    assert float(si) == 0.0 and not sel.any()


def test_batch_scale_and_partial_waves(smpl_set):
    vs, f, ref, _ = smpl_set
    geo = torch.tensor(vs).cuda()
    ref_d = torch.tensor(ref).cuda()
    topo = metric.MeshTopology(f, vs.shape[1])
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    for B in (1, 3 * n_sm + 7, 65536):
        rows = torch.arange(B, device='cuda') % N_SMPL
        v = geo[rows]
        sel = torch.empty(B, len(f), dtype=torch.uint8, device='cuda')
        cnt = topo.counts(v, sel)
        del v
        bad = torch.zeros(B, dtype=torch.bool, device='cuda')
        for r0 in range(0, B, 8192):
            r1 = min(B, r0 + 8192)
            bad[r0:r1] = (sel[r0:r1].bool() != ref_d[rows[r0:r1]]).any(1)
        assert not bad.any(), f'B={B}: rows {torch.nonzero(bad)[:10].flatten().tolist()} differ from the oracle'
        assert torch.equal(cnt.long(), sel.sum(1, dtype=torch.int64)), f'B={B}: counts != selection sums'
        del sel
    torch.cuda.empty_cache()


def test_counts_selection_determinism_nan_row(smpl_set):
    vs, f, ref, _ = smpl_set
    v = torch.tensor(vs[:12]).cuda()
    v[5, int(f[100, 1]), 0] = float('nan')
    v[7, int(f[3, 2]), 2] = float('inf')
    si1, sel1 = metric.self_intersections_percentage(v, torch.tensor(f).cuda(), return_selection=True)
    si2, sel2 = metric.self_intersections_percentage(v, f, return_selection=True)
    assert torch.equal(sel1, sel2) and torch.equal(si1.isnan(), si2.isnan())
    assert torch.equal(si1.nan_to_num(-1), si2.nan_to_num(-1))
    assert torch.equal(sel1.sum(1), torch.round(si1.nan_to_num(0).double() * len(f) / 100).long())
    nan_rows = torch.isnan(si1).cpu().numpy()
    assert nan_rows.tolist() == [r in (5, 7) for r in range(12)]
    assert not sel1[5].any() and not sel1[7].any()
    for r in range(12):
        if r not in (5, 7):
            assert_same(sel1[r].cpu().numpy(), ref[r], vs[r], f, f'row {r}')
            assert float(si1[r]) == np.float32(100.0 * ref[r].sum() / len(f))


def test_cuda_graph_capture_and_replay(smpl_set):
    vs, f, ref, _ = smpl_set
    B = 20
    topo = metric.MeshTopology(f, vs.shape[1])
    v = torch.tensor(vs[:B]).cuda()
    ws = torch.empty(topo.workspace_bytes(B), dtype=torch.uint8, device='cuda')
    sel = torch.zeros(B, len(f), dtype=torch.uint8, device='cuda')
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        topo.counts(v, sel, ws)                           # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        cnt = topo.counts(v, sel, ws)
    v.copy_(torch.tensor(vs[B:2 * B]))
    sel.zero_()
    g.replay()
    torch.cuda.synchronize()
    for r in range(B):
        assert_same(sel[r].cpu().numpy(), ref[B + r], vs[B + r], f, f'graph row {r}')
    assert torch.equal(cnt.long(), torch.tensor(ref[B:2 * B].sum(1)).cuda())


def test_on_body_model_vertices():
    v, f = synthetic.uv_sphere()
    m = synthetic.make_body_tensors('smpl')
    m['v_template'] = torch.tensor(v)
    m['faces'] = torch.tensor(f, dtype=torch.int64)
    B = 6
    bm = BodyModel(m, batch_size=B, model_type='smpl').cuda()
    g = torch.Generator().manual_seed(4)
    with torch.no_grad():
        out = bm(pose_body=0.05 * torch.randn(B, 69, generator=g).cuda())
    verts = out.v
    assert verts.dtype == torch.float32 and verts.is_contiguous() and verts.shape == (B, 6890, 3)
    si, sel = metric.self_intersections_percentage(verts, out.f, return_selection=True)      # faces on the GPU
    host = verts.cpu().numpy()
    for r in range(3):
        assert_same(sel[r].cpu().numpy(), R.selection(host[r], f)[0], host[r], f, f'LBS row {r}')
