"""GPU parity: LBS forward through the C ABI vs the oracle restatement of smplx 0.1.28 (parity unpinned
by the reference: smplx is absent) -- vertices and joints within 1e-5 m (BASELINE.json), plus invariants."""
import pytest
import torch

from dposer_b200 import synthetic
from dposer_b200.body_model import BodyModel, SMPLX
from oracle import lbs_ref

pytestmark = pytest.mark.gpu
TOL_M = 1e-5


def _oracle(model, inputs, mt):
    pose, shape = synthetic.full_pose_from(inputs, mt)
    return lbs_ref.body_forward(model, shape, pose, inputs['trans'])


@pytest.mark.parametrize('mt,B,engine', [('smpl', 1, 1), ('smpl', 37, 1), ('smpl', 256, 1), ('smplx', 1, 1),
                                         ('smplx', 48, 1), ('smpl', 37, 2), ('smpl', 300, 2), ('smplx', 100, 2)])
def test_lbs_forward_vs_oracle(mt, B, engine):
    """engine 1 = fp32 blend, engine 2 = tcgen05 blend (fp16 hi/lo split operands, fp32 accumulate)."""
    m = synthetic.make_body_tensors(mt)
    inp = synthetic.lbs_inputs(B, mt)
    v_ref, j_ref = _oracle(m, inp, mt)
    bm = BodyModel(m, num_betas=10, batch_size=B, model_type=mt).cuda()
    bm.core.engine = engine
    with torch.no_grad():
        out = bm(**{k: v.cuda() for k, v in inp.items()})
    assert out.v.shape == v_ref.shape and out.Jtr.shape == j_ref.shape
    assert (out.v.cpu() - v_ref).abs().max() < TOL_M
    assert (out.Jtr.cpu() - j_ref).abs().max() < TOL_M
    assert out.Jtr.shape[1] == (45 if mt == 'smpl' else 127)
    assert out.full_pose.shape[1] == (72 if mt == 'smpl' else 165)
    # joints-only mode (no vertex output) gives the same joints
    with torch.no_grad():
        out2 = bm(need_verts=False, **{k: v.cuda() for k, v in inp.items()})
    assert out2.v is None
    assert (out2.Jtr - out.Jtr).abs().max() < 5e-6     # extra joints: fp32 blend (compact) vs tcgen05 blend


def test_lbs_large_rotations_and_defaults():
    """Default (omitted) inputs are zeros of batch_size rows; large random rotations everywhere."""
    m = synthetic.make_body_tensors('smpl')
    B = 16
    g = torch.Generator().manual_seed(3)
    pose_body = torch.randn(B, 69, generator=g) * 1.5
    bm = BodyModel(m, batch_size=B, model_type='smpl').cuda()
    with torch.no_grad():
        out = bm(pose_body=pose_body.cuda())
    full = torch.cat([torch.zeros(B, 3), pose_body], 1)
    v_ref, j_ref = lbs_ref.body_forward(m, torch.zeros(B, 10), full, None)
    assert (out.v.cpu() - v_ref).abs().max() < TOL_M
    assert (out.Jtr.cpu() - j_ref).abs().max() < TOL_M
    # zero pose: vertices are the template (betas default to zero)
    with torch.no_grad():
        out0 = bm()
    assert (out0.v.cpu() - m['v_template'][None]).abs().max() < 1e-6


def test_lbs_full_size_batch_properties():
    """Config-2 sized call (65 536 poses) checked through size-independent properties:
    (1) row independence: any row equals the same row computed alone; (2) translation equivariance."""
    m = synthetic.make_body_tensors('smpl')
    B = 65536
    inp = {k: v.cuda() for k, v in synthetic.lbs_inputs(B, 'smpl').items()}
    bm = BodyModel(m, batch_size=B, model_type='smpl').cuda()
    with torch.no_grad():
        out = bm(**inp)
        idx = torch.tensor([0, 1, 4095, 32768, 65535], device='cuda')
        sub = {k: v[idx] for k, v in inp.items()}
        bm_s = BodyModel(m, batch_size=5, model_type='smpl').cuda()
        o2 = bm_s(**sub)
        # the 5-row call takes the fp32 blend, the 65 536-row call the tcgen05 blend: equal to well below 1e-5 m
        assert (out.v[idx] - o2.v).abs().max() < 3e-6 and (out.Jtr[idx] - o2.Jtr).abs().max() < 3e-6
        sub2 = dict(sub)
        sub2['trans'] = sub['trans'] + 1.0
        o3 = bm_s(**sub2)
        assert (o3.v - o2.v - 1.0).abs().max() < 2e-6
    v_ref, j_ref = _oracle(m, {k: v[idx].cpu() for k, v in inp.items()}, 'smpl')
    assert (o2.v.cpu() - v_ref).abs().max() < TOL_M


def test_smplify_wrapper_joints():
    m = synthetic.make_body_tensors('smplx')
    B = 8
    g = torch.Generator().manual_seed(1)
    body = torch.randn(B, 63, generator=g) * 0.3
    glob = torch.randn(B, 3, generator=g)
    betas = torch.randn(B, 10, generator=g)
    transl = torch.randn(B, 3, generator=g)
    smpl = SMPLX(m, batch_size=B).cuda()
    with torch.no_grad():
        out = smpl(betas=betas.cuda(), body_pose=body.cuda(), global_orient=glob.cuda(), transl=transl.cuda())
    # smplx defaults in lib/body_model/smpl.py: hands at the model's constant NON-ZERO mean pose
    full = torch.cat([glob, body, torch.zeros(B, 9), m['hands_mean'][None].expand(B, -1)], 1)
    _, j_ref = lbs_ref.body_forward(m, torch.cat([betas, torch.zeros(B, 10)], 1), full, transl)
    assert out.joints.shape == (B, 49, 3)
    assert (out.joints.cpu() - j_ref[:, smpl.joint_map]).abs().max() < TOL_M


@pytest.mark.parametrize('mt,B,use_verts', [('smpl', 5, True), ('smpl', 19, False), ('smplx', 6, True),
                                            ('smplx', 9, False)])
def test_lbs_backward_vs_autograd_oracle(mt, B, use_verts):
    """dpb_lbs_backward (VJP wrt pose, betas, transl) against torch autograd through the CPU oracle."""
    m = synthetic.make_body_tensors(mt)
    inp = synthetic.lbs_inputs(B, mt, seed=5)
    if mt == 'smplx':   # exercise hands / jaw / eyes too
        g0 = torch.Generator().manual_seed(9)
        inp['pose_hand'] = torch.randn(B, 90, generator=g0) * 0.2
        inp['pose_jaw'] = torch.randn(B, 3, generator=g0) * 0.2
        inp['pose_eye'] = torch.randn(B, 6, generator=g0) * 0.2
        inp['expression'] = torch.randn(B, 10, generator=g0)
    g = torch.Generator().manual_seed(17)
    nj = 45 if mt == 'smpl' else 127
    V = m['v_template'].shape[0]
    gv = torch.randn(B, V, 3, generator=g) / V
    gj = torch.randn(B, nj, 3, generator=g)
    # ---- oracle autograd
    leaf = {k: v.clone().requires_grad_(True) for k, v in inp.items()}
    if mt == 'smpl':
        pose = torch.cat([leaf['root_orient'], leaf['pose_body']], 1)
        shape = leaf['betas']
    else:
        pose = torch.cat([leaf['root_orient'], leaf['pose_body'], leaf['pose_jaw'], leaf['pose_eye'],
                          leaf['pose_hand']], 1)
        shape = torch.cat([leaf['betas'], leaf['expression']], 1)
    v_ref, j_ref = lbs_ref.body_forward(m, shape, pose, leaf['trans'])
    loss = (j_ref * gj).sum() + ((v_ref * gv).sum() if use_verts else 0.0)
    loss.backward()
    # ---- device
    bm = BodyModel(m, num_betas=10, batch_size=B, model_type=mt).cuda()
    dl = {k: v.clone().cuda().requires_grad_(True) for k, v in inp.items()}
    out = bm(need_verts=use_verts, **dl)
    l2 = (out.Jtr * gj.cuda()).sum() + ((out.v * gv.cuda()).sum() if use_verts else 0.0)
    l2.backward()
    for k in inp:
        ref, got = leaf[k].grad, dl[k].grad.cpu()
        scale = ref.abs().max().clamp_min(1e-6)
        err = (got - ref).abs().max() / scale
        assert err < 2e-4, (k, float(err))


@pytest.mark.parametrize('which', ['body_joints_only', 'verts_only'])
def test_lbs_backward_with_an_unused_output(which):
    """Full forward (vertices materialised) but the loss touches one output only, as motion denoising does with
    Jtr[:, :22] (run/motion_denoising.py:236-262): the missing gradient must not be needed (it arrives as None and
    the backward skips the all-vertex pass), and the result must match autograd through the oracle."""
    mt, B = 'smplx', 7
    m = synthetic.make_body_tensors(mt)
    inp = synthetic.lbs_inputs(B, mt, seed=11)
    g = torch.Generator().manual_seed(23)
    V = m['v_template'].shape[0]
    gv = torch.randn(B, V, 3, generator=g) / V
    gj = torch.randn(B, 22, 3, generator=g)
    leaf = {k: v.clone().requires_grad_(True) for k, v in inp.items()}
    zeros = lambda n: torch.zeros(B, n)
    pose = torch.cat([leaf['root_orient'], leaf['pose_body'], zeros(3), zeros(6), zeros(90)], 1)
    shape = torch.cat([leaf['betas'], zeros(10)], 1)
    v_ref, j_ref = lbs_ref.body_forward(m, shape, pose, leaf['trans'])
    ((j_ref[:, :22] * gj).sum() if which == 'body_joints_only' else (v_ref * gv).sum()).backward()
    bm = BodyModel(m, num_betas=10, batch_size=B, model_type=mt).cuda()
    dl = {k: v.clone().cuda().requires_grad_(True) for k, v in inp.items()}
    out = bm(**dl)
    ((out.Jtr[:, :22] * gj.cuda()).sum() if which == 'body_joints_only' else (out.v * gv.cuda()).sum()).backward()
    for k in inp:
        ref, got = leaf[k].grad, dl[k].grad.cpu()
        scale = ref.abs().max().clamp_min(1e-6)
        assert (got - ref).abs().max() / scale < 2e-4, k


@pytest.mark.parametrize('B', [97, 129, 193, 255, 385, 1000])
def test_lbs_pair_kernel_group_boundaries(B):
    """CTA-pair fused kernels: SMPL runs lbs_fused3_kernel (128-pose groups), SMPL-X with the const tail folded into
    the template runs lbs_fused2_kernel (96-pose groups).  Pose counts one past / one short of / straddling groups."""
    for mt in ('smpl', 'smplx'):
        m = synthetic.make_body_tensors(mt)
        inp = synthetic.lbs_inputs(B, mt, seed=17)
        v_ref, j_ref = _oracle(m, inp, mt)
        bm = BodyModel(m, num_betas=10, batch_size=B, model_type=mt).cuda()
        bm.core.engine = 2
        with torch.no_grad():
            out = bm(**{k: v.cuda() for k, v in inp.items()})
        assert (out.v.cpu() - v_ref).abs().max() < TOL_M, mt
        assert (out.Jtr.cpu() - j_ref).abs().max() < TOL_M, mt


def test_smplx_posed_hands_take_the_full_basis_and_const_tail_matches():
    """(1) explicit hand / jaw / eye poses: the const-tail shortcut must NOT be taken (full 486-feature blend);
    (2) SMPLX wrapper (hands at the non-zero mean pose, folded into the template) with vertices, vs the oracle."""
    m = synthetic.make_body_tensors('smplx')
    B = 130
    g = torch.Generator().manual_seed(23)
    inp = synthetic.lbs_inputs(B, 'smplx', seed=19)
    hand, jaw, eye = (0.3 * torch.randn(B, n, generator=g) for n in (90, 3, 6))
    pose = torch.cat([inp['root_orient'], inp['pose_body'], jaw, eye, hand], 1)
    shape = torch.cat([inp['betas'], torch.zeros(B, 10)], 1)
    v_ref, j_ref = lbs_ref.body_forward(m, shape, pose, inp['trans'])
    bm = BodyModel(m, num_betas=10, batch_size=B, model_type='smplx').cuda()
    bm.core.engine = 2
    with torch.no_grad():
        out = bm(pose_hand=hand.cuda(), pose_jaw=jaw.cuda(), pose_eye=eye.cuda(), **{k: v.cuda() for k, v in inp.items()})
    assert (out.v.cpu() - v_ref).abs().max() < TOL_M and (out.Jtr.cpu() - j_ref).abs().max() < TOL_M
    smpl = SMPLX(m, batch_size=B).cuda()
    smpl.core.engine = 2
    with torch.no_grad():
        o2 = smpl(betas=inp['betas'].cuda(), body_pose=inp['pose_body'].cuda(), global_orient=inp['root_orient'].cuda(),
                  transl=inp['trans'].cuda(), need_verts=True)
    full = torch.cat([inp['root_orient'], inp['pose_body'], torch.zeros(B, 9), m['hands_mean'][None].expand(B, -1)], 1)
    v2, j2 = lbs_ref.body_forward(m, shape, full, inp['trans'])
    assert (o2.vertices.cpu() - v2).abs().max() < TOL_M
    assert (o2.joints.cpu() - j2[:, smpl.joint_map]).abs().max() < TOL_M


def test_lbs_fused_kernel_group_boundary_without_translation():
    """tcgen05 engine (fused blend + skinning kernel for SMPL) at a pose count one past a 128-pose group and with no
    translation: the spare joint slot that carries transl must then contribute nothing."""
    m = synthetic.make_body_tensors('smpl')
    B = 129
    inp = synthetic.lbs_inputs(B, 'smpl', seed=13)
    inp.pop('trans')
    pose, shape = synthetic.full_pose_from(inp, 'smpl')
    v_ref, j_ref = lbs_ref.body_forward(m, shape, pose, None)
    bm = BodyModel(m, num_betas=10, batch_size=B, model_type='smpl').cuda()
    bm.core.engine = 2
    with torch.no_grad():
        out = bm(**{k: v.cuda() for k, v in inp.items()})
    assert (out.v.cpu() - v_ref).abs().max() < TOL_M
    assert (out.Jtr.cpu() - j_ref).abs().max() < TOL_M


def test_lbs_backward_split_path_across_tile_boundaries():
    """Vertex cotangents at a batch that crosses the split backward's tiles (8-pose skinning groups, 64-row GEMM tiles,
    128-pose operand padding): gradients must still match autograd through the oracle."""
    mt, B = 'smpl', 70
    m = synthetic.make_body_tensors(mt)
    inp = synthetic.lbs_inputs(B, mt, seed=29)
    g = torch.Generator().manual_seed(31)
    V = m['v_template'].shape[0]
    gv = torch.randn(B, V, 3, generator=g) / V
    gj = torch.randn(B, 45, 3, generator=g)
    leaf = {k: v.clone().requires_grad_(True) for k, v in inp.items()}
    pose = torch.cat([leaf['root_orient'], leaf['pose_body']], 1)
    v_ref, j_ref = lbs_ref.body_forward(m, leaf['betas'], pose, leaf['trans'])
    ((v_ref * gv).sum() + (j_ref * gj).sum()).backward()
    bm = BodyModel(m, num_betas=10, batch_size=B, model_type=mt).cuda()
    dl = {k: v.clone().cuda().requires_grad_(True) for k, v in inp.items()}
    out = bm(**dl)
    ((out.v * gv.cuda()).sum() + (out.Jtr * gj.cuda()).sum()).backward()
    for k in inp:
        ref, got = leaf[k].grad, dl[k].grad.cpu()
        scale = ref.abs().max().clamp_min(1e-6)
        assert (got - ref).abs().max() / scale < 2e-4, k


@pytest.mark.parametrize('mt,B', [('smplx', 96), ('smpl', 130)])
def test_lbs_joints_only_tensor_core_path(mt, B):
    """Joints-only mode (need_verts=False, SMPLify's case) at a batch that takes the tensor-core path: the vertices the
    extra joints / landmarks read run as a small body model of their own (forward AND the backward's vertex pass).
    Joints <= 1e-5 m and gradients <= 2e-4 against autograd through the oracle."""
    m = synthetic.make_body_tensors(mt)
    inp = synthetic.lbs_inputs(B, mt, seed=13)
    nj = 45 if mt == 'smpl' else 127
    gj = torch.randn(B, nj, 3, generator=torch.Generator().manual_seed(29)) * 1e-3
    leaf = {k: v.clone().requires_grad_(True) for k, v in inp.items()}
    if mt == 'smpl':
        pose, shape = torch.cat([leaf['root_orient'], leaf['pose_body']], 1), leaf['betas']
    else:
        pose = torch.cat([leaf['root_orient'], leaf['pose_body'], torch.zeros(B, 99)], 1)
        shape = torch.cat([leaf['betas'], torch.zeros(B, 10)], 1)
    _, j_ref = lbs_ref.body_forward(m, shape, pose, leaf['trans'])
    (j_ref * gj).sum().backward()
    bm = BodyModel(m, num_betas=10, batch_size=B, model_type=mt).cuda()
    dl = {k: v.clone().cuda().requires_grad_(True) for k, v in inp.items()}
    out = bm(need_verts=False, **dl)
    assert out.v is None
    assert float((out.Jtr.detach().cpu() - j_ref.detach()).abs().max()) < 1e-5
    (out.Jtr * gj.cuda()).sum().backward()
    for k in inp:
        ref, got = leaf[k].grad, dl[k].grad.cpu()
        scale = ref.abs().max().clamp_min(1e-12)
        assert float((got - ref).abs().max() / scale) < 2e-4, k


@pytest.mark.parametrize('B', [5, 130])
def test_lbs_interleaved_forwards_keep_their_saved_state(B):
    """A second forward of the same BodyModel between a forward and its backward (gt body / predicted body, as in
    losses.py:251-252) must not disturb the first one's gradient: every differentiable forward owns its workspace."""
    bm = BodyModel(synthetic.make_body_tensors('smplx'), num_betas=10, batch_size=B, model_type='smplx').cuda()
    g = torch.Generator().manual_seed(1)
    pa, pb = torch.randn(B, 63, generator=g).cuda() * 0.3, torch.randn(B, 63, generator=g).cuda() * 0.3
    gv = torch.randn(B, 10475, 3, generator=g).cuda()
    grads = []
    for mode in ('plain', 'nograd_between', 'grad_between'):
        leaf = pa.clone().requires_grad_(True)
        pred = bm(pose_body=leaf)
        if mode == 'nograd_between':
            with torch.no_grad():
                bm(pose_body=pb)
        elif mode == 'grad_between':
            bm(pose_body=pb.clone().requires_grad_(True))
        torch.autograd.backward([pred.v, pred.Jtr], [gv, torch.ones_like(pred.Jtr)])
        grads.append(leaf.grad.clone())
    assert torch.equal(grads[0], grads[1]) and torch.equal(grads[0], grads[2])
