"""Oracle: linear blend skinning -- restatement of third-party smplx==0.1.28.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

**PARITY UNPINNED**: the LBS arithmetic is not in the reference tree; it lives in the
pip dependency ``smplx==0.1.28`` (reference requirements.txt:4; imported at
lib/body_model/body_model.py:4-5 and lib/body_model/smpl.py:3,9-11), which is absent from
this image and cannot be installed offline.  This file restates the published algorithm of
``smplx/lbs.py`` (lbs, blend_shapes, vertices2joints, batch_rodrigues, transform_mat,
batch_rigid_transform) and of ``SMPL.forward`` / ``SMPLX.forward`` / ``VertexJointSelector``
(SURVEY.md Appendix A.6), anchored on the reference's own call sites:
lib/body_model/body_model.py:68-112 and lib/body_model/smpl.py:67-78.  Weak pins available
from the reference: 22-joint parents (lib/body_model/utils.py:180-205), 49-entry joint map
(lib/body_model/smpl.py:53-65), SMPL-X vertex count 10475 (smplx_vert_segmentation.json).
Second opinion: oracle/lbs_np64.py is an independent float64 formulation (no homogeneous matrices); the CPU suite
checks that the two agree to fp32 round-off and that both satisfy the zero-pose / rigid-root / translation /
single-joint invariants (tests/test_oracle_golden.py).
Device-generic: every constant is created on its input's device, so a float64 model dict on CUDA runs there (the
GPU suite's full-batch float64 reference, tests/test_gpu_lbs_scale.py).
"""
import torch

SMPL_PARENTS = [-1, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 9, 12, 13, 14, 16, 17, 18, 19, 20, 21]
SMPLX_PARENTS = SMPL_PARENTS[:22] + [15, 15, 15] + \
    [20, 25, 26, 20, 28, 29, 20, 31, 32, 20, 34, 35, 20, 37, 38] + \
    [21, 40, 41, 21, 43, 44, 21, 46, 47, 21, 49, 50, 21, 52, 53]
# extra vertex joints: nose,reye,leye,rear,lear, 6 feet, 5+5 finger tips (smplx/vertex_ids.py)
SMPL_EXTRA_VIDS = [332, 6260, 2800, 4071, 583, 3216, 3226, 3387, 6617, 6624, 6787,
                   2746, 2319, 2445, 2556, 2673, 6191, 5782, 5905, 6016, 6133]
SMPLX_EXTRA_VIDS = [9120, 9929, 9448, 616, 6, 5770, 5780, 8846, 8463, 8474, 8635,
                    5361, 4933, 5058, 5169, 5286, 8079, 7669, 7794, 7905, 8022]


def batch_rodrigues(rot_vecs):
    """smplx/lbs.py batch_rodrigues: angle = ||r + 1e-8|| (1e-8 added per component)."""
    n = rot_vecs.shape[0]
    angle = torch.norm(rot_vecs + 1e-8, dim=1, keepdim=True)
    rot_dir = rot_vecs / angle
    cos = torch.cos(angle)[:, None]
    sin = torch.sin(angle)[:, None]
    rx, ry, rz = torch.split(rot_dir, 1, dim=1)
    zeros = torch.zeros((n, 1), dtype=rot_vecs.dtype, device=rot_vecs.device)
    K = torch.cat([zeros, -rz, ry, rz, zeros, -rx, -ry, rx, zeros], dim=1).view(n, 3, 3)
    ident = torch.eye(3, dtype=rot_vecs.dtype, device=rot_vecs.device)[None]
    return ident + sin * K + (1 - cos) * torch.bmm(K, K)


def batch_rigid_transform(rot_mats, joints, parents):
    """smplx/lbs.py batch_rigid_transform: chain G_i = G_parent @ [R_i | j_i - j_parent]."""
    B, J = joints.shape[:2]
    joints = joints.unsqueeze(-1)
    rel = joints.clone()
    par = torch.as_tensor(parents[1:], dtype=torch.long, device=joints.device)
    rel[:, 1:] = rel[:, 1:] - joints[:, par]
    top = torch.cat([rot_mats, rel], dim=-1)                              # [B,J,3,4]
    bottom = torch.tensor([0, 0, 0, 1], dtype=joints.dtype, device=joints.device).view(1, 1, 1, 4).expand(B, J, 1, 4)
    M = torch.cat([top, bottom], dim=-2)                                  # [B,J,4,4]
    chain = [M[:, 0]]
    for i in range(1, J):
        chain.append(torch.matmul(chain[parents[i]], M[:, i]))
    G = torch.stack(chain, dim=1)
    posed = G[:, :, :3, 3]
    jh = torch.cat([joints, torch.zeros(B, J, 1, 1, dtype=joints.dtype, device=joints.device)], dim=2)   # [B,J,4,1]
    corr = torch.matmul(G, jh)                                            # [B,J,4,1]
    A = G - torch.nn.functional.pad(corr, [3, 0])
    return posed, A


def lbs(betas, pose, v_template, shapedirs, posedirs, J_regressor, parents, lbs_weights):
    """smplx/lbs.py lbs(pose2rot=True). Returns (verts [B,V,3], posed joints [B,J,3])."""
    B = betas.shape[0]
    J = J_regressor.shape[0]
    v_shaped = v_template[None] + torch.einsum('bl,mkl->bmk', betas, shapedirs)
    Jrest = torch.einsum('bik,ji->bjk', v_shaped, J_regressor)
    R = batch_rodrigues(pose.reshape(-1, 3)).view(B, J, 3, 3)
    feat = (R[:, 1:] - torch.eye(3, dtype=betas.dtype, device=betas.device)).reshape(B, -1)
    v_posed = v_shaped + torch.matmul(feat, posedirs).view(B, -1, 3)
    Jposed, A = batch_rigid_transform(R, Jrest, parents)
    W = lbs_weights[None].expand(B, -1, -1)
    T = torch.matmul(W, A.view(B, J, 16)).view(B, -1, 4, 4)
    vh = torch.cat([v_posed, torch.ones(B, v_posed.shape[1], 1, dtype=betas.dtype, device=betas.device)], dim=2)
    verts = torch.matmul(T, vh.unsqueeze(-1))[:, :, :3, 0]
    return verts, Jposed


def body_forward(model, betas, full_pose, transl=None, chunk=1024):
    """SMPL.forward / SMPLX.forward of smplx 0.1.28 on a synthetic ``model`` dict.

    model keys: v_template[V,3] shapedirs[V,3,S] posedirs[P,3V] J_regressor[J,V] lbs_weights[V,J]
                parents(list) extra_vids(list) and optionally lmk_faces[L,3](vertex ids) lmk_bary[L,3].
    full_pose is the already concatenated [B, J*3] axis-angle pose (pose_mean = 0: BodyModel
    passes flat_hand_mean=True, lib/body_model/body_model.py:30-37).
    joints = cat(lbs joints, verts[:, extra_vids], landmarks) ; + transl on both.
    Chunked over the batch because T=[B,V,4,4] is 441 KB/pose (SURVEY 7 "hard parts").
    """
    vs, js = [], []
    for s in range(0, betas.shape[0], chunk):
        e = s + chunk
        v, j = lbs(betas[s:e], full_pose[s:e], model['v_template'], model['shapedirs'], model['posedirs'],
                   model['J_regressor'], model['parents'], model['lbs_weights'])
        extra = v[:, torch.as_tensor(model['extra_vids'], dtype=torch.long, device=v.device)]
        parts = [j, extra]
        if model.get('lmk_faces') is not None:
            tri = v[:, model['lmk_faces'].reshape(-1)].view(v.shape[0], -1, 3, 3)
            parts.append(torch.einsum('blfi,lf->bli', tri, model['lmk_bary']))
        j = torch.cat(parts, dim=1)
        if transl is not None:
            j = j + transl[s:e, None]
            v = v + transl[s:e, None]
        vs.append(v)
        js.append(j)
    return torch.cat(vs), torch.cat(js)
