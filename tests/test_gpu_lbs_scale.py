"""LBS forward and backward at the batch sizes the benchmark and the fitting loops run, every row against the float64
restatement of smplx (oracle/lbs_ref.py, run on the GPU in batch chunks), plus a direct test of the motion-denoising
loss kernel (dpb_motion_loss) against a float64 restatement of run/motion_denoising.py:255-262.

Forward: max |got - ref| over every vertex and joint of every row <= 1e-5 m (BASELINE.json).
Backward: vector-Jacobian products against float64 autograd with the same cotangents, per row and per output:
max |got - ref| / max |ref of that row| <= 2e-4; rows whose cotangents are all zero must get exactly zero gradients.
"""
import ctypes
import math
import types

import pytest
import torch

from dposer_b200 import _lib as L
from dposer_b200 import steps as S
from dposer_b200 import synthetic
from dposer_b200.body_model import BodyModel, SMPLX
from oracle import lbs_ref

pytestmark = pytest.mark.gpu
TOL_M = 1e-5
TOL_G = 2e-4
NP_FUSED3 = 128          # poses per group of lbs_fused3_kernel
TILE_PAIR = 256          # vertices per CTA-pair tile of lbs_fused3_kernel


@pytest.fixture(scope='module')
def body():
    """Synthetic SMPL / SMPL-X body tensors (fp32, host) and their float64 copies on cuda:0 for the reference."""
    out = {}
    for mt in ('smpl', 'smplx'):
        m = synthetic.make_body_tensors(mt)
        m64 = {k: (v.cuda().double() if v.is_floating_point() else v.cuda()) if torch.is_tensor(v) else v
               for k, v in m.items()}
        out[mt] = (m, m64)
    return out


def _forward_only(core, B, need_verts=True):
    """An LbsStep for forward-only calls: built with need_verts=False (no vertex cotangents, no all-vertex backward
    scratch), then given a vertex output of its own unless joints-only.  Outputs start as NaN so a row the kernel never
    writes cannot pass."""
    lbs = S.LbsStep(core, B, 'cuda', need_verts=False)
    lbs.verts = torch.full((B, core.V, 3), float('nan'), device='cuda') if need_verts else None
    lbs.joints.fill_(float('nan'))
    return lbs


def _ref_chunks(m64, shape, pose, transl, chunk, grad=False):
    """(s, e, leaves, verts, joints) of the float64 reference, chunk by chunk (peak memory of one chunk)."""
    B = shape.shape[0]
    for s in range(0, B, chunk):
        e = min(B, s + chunk)
        leaves = [x[s:e].double().requires_grad_(grad) if x is not None else None for x in (shape, pose, transl)]
        with torch.set_grad_enabled(grad):
            v, j = lbs_ref.body_forward(m64, leaves[0], leaves[1], leaves[2], chunk=e - s)
        yield s, e, leaves, v, j


class _RowMax:
    """Largest error of every row, and where it is, for the report of a failing forward."""

    def __init__(self, B, device='cuda'):
        self.err = torch.zeros(B, dtype=torch.float64, device=device)
        self.arg = torch.zeros(B, dtype=torch.long, device=device)

    def add(self, s, got, ref):
        d = (got.double() - ref).abs().amax(dim=2)          # [n, points]
        self.err[s:s + d.shape[0]], self.arg[s:s + d.shape[0]] = d.max(dim=1)

    def check(self, what, tol=TOL_M):
        worst = float(self.err.max())
        print(f'[lbs-scale] {what}: max |d| = {worst:.3e} m')
        if not worst <= tol:
            bad = torch.nonzero(~(self.err <= tol)).flatten()
            rows = [(int(r), int(self.arg[r]), float(self.err[r])) for r in bad[:20]]
            raise AssertionError(f'{what}: {bad.numel()} rows above {tol:g} m; (row, point, err) = {rows}')
        return worst


def _check_forward(m64, shape, pose, transl, verts, joints, what, chunk=1024):
    B = shape.shape[0]
    ev = _RowMax(B) if verts is not None else None
    ej = _RowMax(B)
    for s, e, _, v, j in _ref_chunks(m64, shape, pose, transl, chunk):
        if ev is not None:
            ev.add(s, verts[s:e], v)
        ej.add(s, joints[s:e], j)
    if ev is not None:
        ev.check(what + ' vertices')
    ej.check(what + ' joints')


# ------------------------------------------------------------------------------------------------------------------
# the float64 reference itself on the GPU


@pytest.mark.parametrize('mt', ['smpl', 'smplx'])
def test_float64_reference_same_on_cuda_and_cpu(body, mt):
    """lbs_ref.body_forward in float64 gives the same vertices, joints and autograd gradients on CUDA and on CPU."""
    m, m64 = body[mt]
    m64cpu = {k: (v.double() if v.is_floating_point() else v) if torch.is_tensor(v) else v for k, v in m.items()}
    B = 5
    inp = synthetic.lbs_inputs(B, mt, seed=3)
    pose, shape = synthetic.full_pose_from(inp, mt)
    g = torch.Generator().manual_seed(4)
    pose = pose + 0.3 * torch.randn(pose.shape, generator=g)          # hands / jaw / eyes posed too
    gv = torch.randn(B, m['v_template'].shape[0], 3, generator=g, dtype=torch.float64)
    gj = torch.randn(B, 45 if mt == 'smpl' else 127, 3, generator=g, dtype=torch.float64)
    res = []
    for model, dev in ((m64cpu, 'cpu'), (m64, 'cuda')):
        leaves = [x.double().to(dev).requires_grad_(True) for x in (shape, pose, inp['trans'])]
        v, j = lbs_ref.body_forward(model, *leaves)
        ((v * gv.to(dev)).sum() + (j * gj.to(dev)).sum()).backward()
        res.append([v.detach().cpu(), j.detach().cpu()] + [x.grad.cpu() for x in leaves])
    for a, b in zip(*res):
        assert float((a - b).abs().max()) <= 1e-12 * max(1.0, float(b.abs().max()))


# ------------------------------------------------------------------------------------------------------------------
# forward


def test_smpl_forward_65536_every_row(body, monkeypatch):
    """Config 2 (65 536 SMPL poses, AUTO engine: lbs_fused3_kernel): every vertex and joint of every row <= 1e-5 m;
    the forward-only call (no saved transforms, what BodyModel does under no_grad), the saving call (what it does when
    an input requires grad) and the call with both L2 cache hints off (DPB_LBS_DEBUG=48) are bit-identical."""
    m, m64 = body['smpl']
    B = 65536
    inp = {k: v.cuda() for k, v in synthetic.lbs_inputs(B, 'smpl', seed=41).items()}
    pose, shape = synthetic.full_pose_from(inp, 'smpl')
    pose, shape, transl = pose.contiguous(), shape.contiguous(), inp['trans'].contiguous()
    core = BodyModel(m, batch_size=B, model_type='smpl').cuda().core
    a = _forward_only(core, B)
    a.forward(shape, pose, transl, no_save=True)
    b = _forward_only(core, B)
    b.forward(shape, pose, transl, no_save=False)
    assert torch.equal(a.verts, b.verts) and torch.equal(a.joints, b.joints)
    del b
    monkeypatch.setenv('DPB_LBS_DEBUG', '48')
    c = _forward_only(core, B)
    c.forward(shape, pose, transl, no_save=True)
    assert torch.equal(a.verts, c.verts) and torch.equal(a.joints, c.joints)
    del c
    _check_forward(m64, shape, pose, transl, a.verts, a.joints, 'smpl B=65536')


def _fused3_split(V):
    """lbs_fused3's work split for a V-vertex model: ceil(B/128) pose groups x n_tp tile pairs (vertices padded to whole
    pairs of 128-vertex tiles) over sm_count/2 CTA pairs.  Returns (workers, n_tp, the batches that change the split)."""
    sm = ctypes.c_int()
    L.check(L.load().dpb_device_info(0, ctypes.byref(sm), None, None))
    workers = (sm.value & ~1) // 2
    n_tp = (V + TILE_PAIR - 1) // TILE_PAIR
    groups = max(g for g in range(1, 65536 // NP_FUSED3 + 1) if (g * n_tp) % workers == 0)
    return workers, n_tp, {'exact_multiple': groups * NP_FUSED3, 'plus_one': groups * NP_FUSED3 + 1, '65535': 65535}


@pytest.mark.parametrize('which', ['exact_multiple', 'plus_one', '65535'])
def test_smpl_forward_fused3_worker_splits(body, which):
    """Every row at a batch whose item count is a whole multiple of the worker count (every worker ends on a tile-pair
    boundary), one pose past it (a partial last group, uneven split), and 65 535 (a partial last group at full size)."""
    m, m64 = body['smpl']
    core = BodyModel(m, model_type='smpl').cuda().core
    workers, n_tp, batches = _fused3_split(core.V)
    B = batches[which]
    items = (B + NP_FUSED3 - 1) // NP_FUSED3 * n_tp
    assert (items % workers == 0) == (which == 'exact_multiple'), (B, items, workers)
    inp = {k: v.cuda() for k, v in synthetic.lbs_inputs(B, 'smpl', seed=43).items()}
    pose, shape = synthetic.full_pose_from(inp, 'smpl')
    pose, shape, transl = pose.contiguous(), shape.contiguous(), inp['trans'].contiguous()
    lbs = _forward_only(core, B)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        lbs.forward(shape, pose, transl, no_save=True)
        torch.cuda.synchronize()
    assert any('lbs_fused3_kernel' in e.name for e in prof.events()), 'the split under test is lbs_fused3_kernel\'s'
    _check_forward(m64, shape, pose, transl, lbs.verts, lbs.joints, f'smpl B={B} ({which})')


# ------------------------------------------------------------------------------------------------------------------
# backward


def _mixed_factors(B, seed):
    """Per-row cotangent factors 2^k, k in [-40, 10]; every 16th row (from a seeded offset) exactly zero."""
    g = torch.Generator().manual_seed(seed)
    k = torch.randint(-40, 11, (B,), generator=g)
    f = torch.pow(2.0, k.double())
    f[int(torch.randint(16, (1,), generator=g)):: 16] = 0.0
    return f.cuda()


def _single_vertex(gv, gj, row, vid):
    """Keep the cotangent of one vertex of ``row`` only."""
    keep = gv[row, vid].clone()
    gv[row].zero_()
    gv[row, vid] = keep
    if gj is not None:
        gj[row].zero_()


def _nan_grads(lbs):
    """Gradient outputs start as NaN, so a row the backward never writes cannot pass (nor keep an earlier result)."""
    for t in (lbs.g_pose, lbs.g_shape, lbs.g_transl):
        t.fill_(float('nan'))


class _RowGrad:
    """Per-row relative error of one gradient output: max |got - ref| / max |ref of that row|."""

    def __init__(self, name):
        self.name, self.worst, self.where = name, 0.0, None

    def add(self, s, got, ref):
        got, ref = got.double().reshape(got.shape[0], -1), ref.double().reshape(ref.shape[0], -1)
        den = ref.abs().amax(1)
        zero = den == 0
        if bool(zero.any()):
            nz = (got[zero] != 0).any(1)
            assert not bool(nz.any()), f'{self.name}: rows {(torch.nonzero(zero).flatten()[nz] + s).tolist()[:10]} ' \
                                       'have zero cotangents but non-zero gradients'
        if bool((~zero).any()):
            rel = (got - ref).abs().amax(1)[~zero] / den[~zero]
            r = float(rel.max())
            if math.isnan(r) or r > self.worst:      # a NaN stays the worst (it compares False with anything)
                self.worst, self.where = r, s + int(torch.nonzero(~zero).flatten()[rel.argmax()])

    def check(self, what):
        print(f'[lbs-scale] {what} {self.name}: per-row max rel err = {self.worst:.3e} (row {self.where})')
        assert self.worst <= TOL_G, (what, self.name, self.worst, self.where)


def _check_vjp(m64, shape, pose, transl, gv, gj, got, what, chunk, factors=None, mixed=None, forward=None):
    """Float64 autograd VJP with cotangents (gv, gj), chunk by chunk, against the device gradients ``got``
    (g_pose, g_shape[, g_transl]).  ``factors`` / ``mixed``: a second device result for the cotangents scaled per row
    (its reference is the same VJP scaled: the VJP is linear).  ``forward`` = (verts, joints) also checks the forward."""
    names = ['g_pose', 'g_betas', 'g_transl'][:len(got)]
    acc = [_RowGrad(n) for n in names]
    acc_m = [_RowGrad(n) for n in names]
    fv = _RowMax(shape.shape[0]) if forward is not None and forward[0] is not None else None
    fj = _RowMax(shape.shape[0]) if forward is not None else None
    for s, e, leaves, v, j in _ref_chunks(m64, shape, pose, transl, chunk, grad=True):
        if fv is not None:
            fv.add(s, forward[0][s:e], v.detach())
        if fj is not None:
            fj.add(s, forward[1][s:e], j.detach())
        loss = (j * gj[s:e].double()).sum()
        if gv is not None:
            loss = loss + (v * gv[s:e].double()).sum()
        ins = [leaves[0], leaves[1]] + ([leaves[2]] if len(got) > 2 else [])
        refs = torch.autograd.grad(loss, ins)
        refs = [refs[1], refs[0]] + list(refs[2:])       # (pose, shape, transl) order of `got`
        for a, g, r in zip(acc, got, refs):
            a.add(s, g[s:e], r)
        if mixed is not None:
            for a, g, r in zip(acc_m, mixed, refs):
                a.add(s, g[s:e], r * factors[s:e, None])
        del loss, refs, v, j
    if fv is not None:
        fv.check(what + ' vertices')
    if fj is not None:
        fj.check(what + ' joints')
    for a in acc:
        a.check(what)
    if mixed is not None:
        for a in acc_m:
            a.check(what + ' mixed-magnitude')


def test_config4_smplx_backward_motion_cotangents(body):
    """Config 4 (motion denoising: 256 sequences x 60 frames of SMPL-X, hands / jaw / eyes at the constant zero tail):
    the forward of MotionDenoise's LbsStep (96-pose-group kernel, DPB_LBS_CONST_TAIL) on every row, then the backward
    with the vertex and joint cotangents that dpb_motion_loss computes from those vertices (the pipeline's scale,
    ~w / ((L-1) V)), then with the same cotangents scaled per row by 2^k (zero rows, one single-vertex row)."""
    m, m64 = body['smplx']
    seq_len, n_seq = 60, 256
    B = seq_len * n_seq
    pose, shape = synthetic.full_pose_from(synthetic.lbs_inputs(B, 'smplx', seed=47), 'smplx')
    pose, shape = pose.cuda().contiguous(), shape.cuda().contiguous()
    core = BodyModel(m, num_betas=10, batch_size=B, model_type='smplx').cuda().core
    lbs = S.LbsStep(core, B, 'cuda', need_verts=True)
    lbs.verts.fill_(float('nan'))
    lbs.joints.fill_(float('nan'))
    lbs.forward(shape, pose, None)
    g = torch.Generator(device='cuda').manual_seed(5)
    target = (lbs.joints[:, :22] + 0.04 * torch.randn(B, 22, 3, generator=g, device='cuda')).contiguous()
    S.motion_loss(lbs, target, seq_len, 22, 10.0, 100.0)
    gv, gj = lbs.g_verts.clone(), lbs.g_joints.clone()
    _nan_grads(lbs)
    lbs.backward(shape, pose, use_verts=True)
    got = [lbs.g_pose.clone(), lbs.g_shape.clone()]
    f = _mixed_factors(B, 6)
    row1 = int(torch.nonzero(f).flatten()[7])
    lbs.g_verts.mul_(f[:, None, None].float())
    lbs.g_joints.mul_(f[:, None, None].float())
    _single_vertex(lbs.g_verts, lbs.g_joints, row1, 5000)
    gv1, gj1 = lbs.g_verts[row1:row1 + 1].clone(), lbs.g_joints[row1:row1 + 1].clone()
    _nan_grads(lbs)
    lbs.backward(shape, pose, use_verts=True)
    mixed = [lbs.g_pose.clone(), lbs.g_shape.clone()]
    one = [x[row1:row1 + 1].clone() for x in mixed]
    for x in mixed:
        x[row1] = 0.0
    f[row1] = 0.0
    _check_vjp(m64, shape, pose, None, gv, gj, got, 'config4 smplx B=15360', 256, f, mixed,
               forward=(lbs.verts, lbs.joints))
    one_row = slice(row1, row1 + 1)
    _check_vjp(m64, shape[one_row], pose[one_row], None, gv1, gj1, one, 'config4 single-vertex row', 1)


def test_config5_smplx_joints_only_131072(body):
    """Config 5 (SMPLify: 131 072 SMPL-X rows, joints only, hands at the model's constant mean pose): forward with and
    without saving (bit-identical, all n_out joints <= 1e-5 m), then the backward with joint cotangents only through
    the tensor-core compact-vertex pass, with unit-scale and per-row 2^k-scaled cotangents (zero rows included)."""
    m, m64 = body['smplx']
    B = 131072
    smpl = SMPLX(m, batch_size=B).cuda()
    core = smpl.core
    inp = {k: v.cuda() for k, v in synthetic.lbs_inputs(B, 'smplx', seed=53).items()}
    pose = torch.zeros(B, core.J * 3, device='cuda')
    pose[:, :66] = torch.cat([inp['root_orient'], inp['pose_body']], 1)
    pose[:, 75:] = smpl.hand_mean
    shape = torch.zeros(B, core.S, device='cuda')
    shape[:, :10] = inp['betas']
    transl = inp['trans'].contiguous()
    a = _forward_only(core, B, need_verts=False)
    a.forward(shape, pose, transl, no_save=True)
    lbs = S.LbsStep(core, B, 'cuda', need_verts=False)
    lbs.joints.fill_(float('nan'))
    lbs.forward(shape, pose, transl, no_save=False)
    assert torch.equal(a.joints, lbs.joints)
    del a
    g = torch.Generator(device='cuda').manual_seed(7)
    gj = torch.randn(B, core.n_out, 3, generator=g, device='cuda')
    lbs.g_joints.copy_(gj)
    _nan_grads(lbs)
    lbs.backward(shape, pose, use_verts=False, want_transl=True)
    got = [lbs.g_pose.clone(), lbs.g_shape.clone(), lbs.g_transl.clone()]
    f = _mixed_factors(B, 8)
    lbs.g_joints.mul_(f[:, None, None].float())
    _nan_grads(lbs)
    lbs.backward(shape, pose, use_verts=False, want_transl=True)
    mixed = [lbs.g_pose.clone(), lbs.g_shape.clone(), lbs.g_transl.clone()]
    _check_vjp(m64, shape, pose, transl, None, gj, got, 'config5 smplx B=131072', 512, f, mixed,
               forward=(None, lbs.joints))


def test_smpl_backward_4096_mixed_magnitudes(body):
    """SMPL at 4 096 rows with vertex, joint and translation gradients (the split tensor-core backward): unit-scale
    cotangents, then per-row 2^k-scaled ones with zero rows and one row whose only cotangent is on a single vertex."""
    m, m64 = body['smpl']
    B = 4096
    inp = {k: v.cuda() for k, v in synthetic.lbs_inputs(B, 'smpl', seed=59).items()}
    pose, shape = synthetic.full_pose_from(inp, 'smpl')
    pose, shape, transl = pose.contiguous(), shape.contiguous(), inp['trans'].contiguous()
    core = BodyModel(m, batch_size=B, model_type='smpl').cuda().core
    lbs = S.LbsStep(core, B, 'cuda', need_verts=True)
    lbs.forward(shape, pose, transl)
    g = torch.Generator(device='cuda').manual_seed(9)
    gv = torch.randn(B, core.V, 3, generator=g, device='cuda') / core.V
    gj = torch.randn(B, core.n_out, 3, generator=g, device='cuda')
    lbs.g_verts.copy_(gv)
    lbs.g_joints.copy_(gj)
    _nan_grads(lbs)
    lbs.backward(shape, pose, use_verts=True, want_transl=True)
    got = [lbs.g_pose.clone(), lbs.g_shape.clone(), lbs.g_transl.clone()]
    f = _mixed_factors(B, 10)
    row1 = int(torch.nonzero(f).flatten()[3])
    lbs.g_verts.mul_(f[:, None, None].float())
    lbs.g_joints.mul_(f[:, None, None].float())
    _single_vertex(lbs.g_verts, lbs.g_joints, row1, 1234)
    gv1, gj1 = lbs.g_verts[row1:row1 + 1].clone(), lbs.g_joints[row1:row1 + 1].clone()
    _nan_grads(lbs)
    lbs.backward(shape, pose, use_verts=True, want_transl=True)
    mixed = [lbs.g_pose.clone(), lbs.g_shape.clone(), lbs.g_transl.clone()]
    one = [x[row1:row1 + 1].clone() for x in mixed]
    for x in mixed:
        x[row1] = 0.0
    f[row1] = 0.0
    _check_vjp(m64, shape, pose, transl, gv, gj, got, 'smpl B=4096', 1024, f, mixed)
    one_row = slice(row1, row1 + 1)
    _check_vjp(m64, shape[one_row], pose[one_row], transl[one_row], gv1, gj1, one, 'smpl single-vertex row', 1)


# ------------------------------------------------------------------------------------------------------------------
# dpb_motion_loss


def _motion_ref(verts, joints, target, seq_len, n_data, w_temp, w_data):
    """Float64 restatement of run/motion_denoising.py:255-262 applied per sequence: temporal term
    mean_{t,v} ||v[t] - v[t+1]||, data term mean_{t,j<n_data} ||J[t,j] - target[t,j]|| (dropped unless > 0, so NaN and
    0 drop it), their per-sequence values and the cotangents of w_temp * temp + w_data * data.  A zero distance has a
    zero cotangent (the kernel's choice where sqrt's derivative is undefined)."""
    n_seq = verts.shape[0] // seq_len
    V, n_out = verts.shape[1], joints.shape[1]
    v = verts.double().view(n_seq, seq_len, V, 3)
    d = v[:, :-1] - v[:, 1:]
    dn = d.norm(dim=3, keepdim=True)
    temp = dn.mean(dim=(1, 2, 3))
    u = torch.where(dn > 0, d / dn, torch.zeros_like(d)) * (w_temp / ((seq_len - 1) * V))
    gv = torch.zeros_like(v)
    gv[:, :-1] += u
    gv[:, 1:] -= u
    e = joints.double().view(n_seq, seq_len, n_out, 3)[:, :, :n_data] - target.double().view(n_seq, seq_len, n_data, 3)
    en = e.norm(dim=3, keepdim=True)
    data = en.mean(dim=(1, 2, 3))
    gj = torch.zeros(n_seq, seq_len, n_out, 3, dtype=torch.float64, device=verts.device)
    gj[:, :, :n_data] = torch.where(en > 0, e / en, torch.zeros_like(e)) * (w_data / (seq_len * n_data))
    gj[~(data > 0)] = 0.0
    return torch.stack([temp, data], 1), gv.view(-1, V, 3), gj.view(-1, n_out, 3)


def _motion_run(verts, joints, target, seq_len, n_data, w_temp=10.0, w_data=100.0):
    rows, V, n_out = verts.shape[0], verts.shape[1], joints.shape[1]
    lbs = types.SimpleNamespace(verts=verts, joints=joints, rows=rows, dev=verts.device,
                                core=types.SimpleNamespace(V=V, n_out=n_out),
                                g_verts=torch.full_like(verts, float('nan')), g_joints=torch.full_like(joints, float('nan')))
    terms = torch.full((rows // seq_len, 2), float('nan'), device=verts.device)
    S.motion_loss(lbs, target, seq_len, n_data, w_temp, w_data, seq_terms=terms)
    return terms, lbs.g_verts, lbs.g_joints


def _nanmax(a, b):
    return a if math.isnan(a) else (b if math.isnan(b) or b > a else a)


def _motion_check(verts, joints, target, seq_len, n_data, seq_chunk=32):
    """Kernel vs the float64 reference, sequence by sequence: cotangents to 1e-6 of the sequence's largest, the data
    term to 1e-5 relative (block sum in fp32), the temporal term to 1e-5 relative (fp32 atomics)."""
    terms, g_v, g_j = _motion_run(verts, joints, target, seq_len, n_data)
    assert not bool(torch.isnan(g_v).any()) and not bool(torch.isnan(g_j).any())
    assert bool((g_j[:, n_data:] == 0).all())
    n_seq = verts.shape[0] // seq_len
    worst = [0.0, 0.0, 0.0]
    for s0 in range(0, n_seq, seq_chunk):
        s1 = min(n_seq, s0 + seq_chunk)
        r0, r1 = s0 * seq_len, s1 * seq_len
        t_ref, gv_ref, gj_ref = _motion_ref(verts[r0:r1], joints[r0:r1], target[r0:r1], seq_len, n_data, 10.0, 100.0)
        for i, (got, ref) in enumerate(((g_v[r0:r1], gv_ref), (g_j[r0:r1], gj_ref))):
            got = got.double().view(s1 - s0, -1)
            ref = ref.view(s1 - s0, -1)
            den = ref.abs().amax(1)
            err = (got - ref).abs().amax(1)
            assert bool((err[den == 0] == 0).all()), 'a dropped / zero sequence got a non-zero cotangent'
            rel = err[den > 0] / den[den > 0]
            if rel.numel():
                worst[i] = _nanmax(worst[i], float(rel.max()))
        tt = terms[s0:s1].double()
        nan = torch.isnan(t_ref)
        assert torch.equal(torch.isnan(tt), nan)
        rel = ((tt - t_ref).abs() / t_ref.abs().clamp_min(1e-30))[~nan]
        worst[2] = _nanmax(worst[2], float(rel.max()))
    print(f'[motion-loss] L={seq_len}: g_verts {worst[0]:.2e}, g_joints {worst[1]:.2e}, seq_terms {worst[2]:.2e}')
    assert worst[0] <= 1e-6 and worst[1] <= 1e-6 and worst[2] <= 1e-5, worst
    return terms, g_v, g_j


def _motion_inputs(n_seq, seq_len, V=10475, n_out=127, n_data=22, seed=61):
    g = torch.Generator(device='cuda').manual_seed(seed)
    rows = n_seq * seq_len
    base = torch.rand(n_seq, 1, V, 3, generator=g, device='cuda') - 0.5
    walk = 0.01 * torch.randn(n_seq, seq_len, V, 3, generator=g, device='cuda')
    verts = (base + walk.cumsum(1)).reshape(rows, V, 3).contiguous()
    joints = torch.randn(rows, n_out, 3, generator=g, device='cuda') * 0.5
    target = (joints[:, :n_data] + 0.04 * torch.randn(rows, n_data, 3, generator=g, device='cuda')).contiguous()
    return verts, joints, target


def test_motion_loss_vs_float64_edges():
    """256 sequences x 60 frames, V = 10 475 (not a multiple of 128), n_out = 127, n_data = 22, with: a sequence whose
    joints equal their target (data term 0: dropped for that sequence only), one with a NaN target (dropped, no NaN in
    any cotangent), repeated frames / a joint exactly on its target (zero distance: zero cotangent), then sequence
    independence: perturbing the last frame of one sequence changes that sequence's terms and cotangents only."""
    seq_len, n_seq, n_data = 60, 256, 22
    verts, joints, target = _motion_inputs(n_seq, seq_len)
    r = lambda s, f=0: s * seq_len + f          # noqa: E731
    target[r(3):r(4)] = joints[r(3):r(4), :n_data]                 # sequence 3: data term exactly 0
    target[r(9, 17), 4, 1] = float('nan')                          # sequence 9: NaN target
    verts[r(5, 11)] = verts[r(5, 10)]                              # sequence 5: a repeated frame
    verts[r(6, 0):r(6, 5)] = verts[r(6, 0)]                        # sequence 6: five equal frames
    target[r(7, 2), 0] = joints[r(7, 2), 0]                        # sequence 7: one joint exactly on target
    terms, g_v, g_j = _motion_check(verts, joints, target, seq_len, n_data)
    assert float(terms[3, 1]) == 0.0 and bool((g_j[r(3):r(4)] == 0).all())
    assert bool(torch.isnan(terms[9, 1])) and bool((g_j[r(9):r(10)] == 0).all())
    assert bool((g_j[r(8):r(9), :n_data] != 0).any()) and bool((g_j[r(10):r(11), :n_data] != 0).any())
    assert bool((g_j[r(7, 2), 0] == 0).all())
    # sequence independence
    s = 100
    verts[r(s, seq_len - 1)] += 0.05
    joints[r(s, seq_len - 1)] += 0.05
    t2, gv2, gj2 = _motion_run(verts, joints, target, seq_len, n_data)
    for a, b in ((gv2, g_v), (gj2, g_j)):
        assert torch.equal(a[:r(s)], b[:r(s)]) and torch.equal(a[r(s + 1):], b[r(s + 1):])
        assert not torch.equal(a[r(s, seq_len - 1)], b[r(s, seq_len - 1)])
    assert not torch.equal(gv2[r(s, seq_len - 2)], g_v[r(s, seq_len - 2)])
    other = torch.ones(n_seq, dtype=torch.bool, device='cuda')
    other[s] = False
    assert torch.equal(t2[other, 1].nan_to_num(), terms[other, 1].nan_to_num())     # (sequence 9's term is NaN)
    # the temporal term is summed with fp32 atomics: another run may order them differently (last bits only)
    assert float(((t2[other, 0] - terms[other, 0]).abs() / terms[other, 0].abs()).max()) <= 1e-5
    assert float(t2[s, 0]) != float(terms[s, 0]) and float(t2[s, 1]) != float(terms[s, 1])


def test_motion_loss_two_frame_sequences():
    """seq_len = 2: one difference per sequence; the first and last frame carry opposite cotangents."""
    verts, joints, target = _motion_inputs(96, 2, seed=67)
    _, g_v, _ = _motion_check(verts, joints, target, 2, 22)
    assert torch.equal(g_v[0::2], -g_v[1::2])
