"""Metrics of the hot path as device reductions (reference lib/utils/metric.py:8-89 and
lib/dataset/AMASS.py:263-324).  ``average_pairwise_distance`` runs on one GPU unless the caller opts into
sharding with an explicit ``group=`` (then every rank of the group must call it).

Self-intersection metric SI (``self_intersections_percentage``)
----------------------------------------------------------------
The reference (lib/utils/metric.py:41-89) selects self-intersecting faces with pymeshlab, i.e. VCG's
``Clean::SelfIntersections`` and its ``TestFaceFaceIntersection``, one mesh at a time on the CPU.  Parity with
pymeshlab is unpinned; the rule below follows that code as far as it is known and is this project's definition.

For one mesh with vertices ``P [V,3]`` (fp32) and faces ``F [nF,3]`` (int), a pair of distinct faces (f, g)
**intersects** according to ``s``, the number of vertex ids the two faces share:

- **s = 0**: the two *closed* triangles have a common point. This includes touching at a vertex or edge, and
  coplanar overlap.
- **s = 1**: let v be the shared vertex. The segment joining the midpoints of f's two edges at v crosses the *open
  interior* of g: the segment's endpoints lie strictly on opposite sides of g's plane, and all three barycentric
  coordinates of the crossing point are > 0. The same test is also run with f and g swapped. Either one passing is
  enough. This is VCG's "opposite edge moved halfway to the shared vertex".
- **s = 2** (faces sharing an edge, i.e. a fold): never counted.
- **s = 3** (the same three vertex ids): counted.
- A face with zero area never intersects anything.

A face is **selected** if it belongs to at least one intersecting pair. ``SI = 100 · (selected faces) / nF``. If a
face references a vertex with a non-finite coordinate, that mesh's SI is NaN and its selection is all false. Other
meshes in the batch are unaffected.

Every decision is a sign of an fp64 expression evaluated on the fp32 inputs. The oracle and the kernel use the same
formulas. Any fp32 pre-filter in the kernel, such as AABB or plane-side rejection, must be conservative: it may keep a
pair that the exact test rejects, but never the reverse.

The formulas (``csrc/selfisect.cu``, restated in ``oracle/selfisect_ref.py``): n = (q1 - q0) x (q2 - q0) is a face's
normal (zero area: n == 0 exactly); s = 0 holds when an edge of either face meets the other closed triangle -- the
edge's end points relative to the plane, n . (x - q0), then either the three signed volumes (b - a) . ((q_i - a) x
(q_i+1 - a)) all >= 0 or all <= 0, or, for an edge in the plane, in-plane orientations n . ((q - p) x (r - p)) and
on-segment dot products; s = 1 uses the same volumes, strictly.  Both implementations also require the closed fp32
AABBs of the two faces to overlap, an exact test that no intersecting pair fails.

Procrustes-aligned point error PA-MPJPE / PA-MPVPE (``compute_similarity_transform``, ``reconstruction_error``)
------------------------------------------------------------------------------------------------------------
The reference computes it in lib/utils/transforms.py with numpy, one sample at a time; that file is not part of the
checkout this was built from, so parity is unpinned and the rule is this project's: the similarity Procrustes with the
reflection correction, as in HMR / SPIN's ``compute_similarity_transform``.  For one sample with predicted points
``S1 [n,3]`` and target points ``S2 [n,3]`` (fp32 inputs, evaluated in float64)::

    mu1, mu2 = mean(S1), mean(S2);  X1 = S1 - mu1;  X2 = S2 - mu2
    var1 = sum(X1**2);  K = X1^T X2                      # 3x3
    U, s, Vh = svd(K);  V = Vh^T
    Z = diag(1, 1, sign(det(U V^T)))                     # det is +-1, never 0
    R = V Z U^T;  scale = trace(R K) / var1;  t = mu2 - scale R mu1
    S1_hat = scale S1 R^T + t                            # row-vector form
    err = mean_k ||S1_hat[k] - S2[k]||                   # in the input's units (metres)

- **Subset.** An optional point subset ``idx`` selects the points that both fit the transform and are measured;
  ``S1_hat`` applies that transform to all ``n`` points.
- **NaN rows.** A row whose selected points hold a non-finite coordinate gets NaN for ``err``, its parameters and its
  aligned points; so does a row with ``var1 == 0`` (all selected predicted points coincide, or one point).  A
  non-finite coordinate outside the subset only makes its own aligned point non-finite.  Other rows are unaffected.
- **Uniqueness.** ``R`` is unique when the smallest singular value of ``K`` is simple (coplanar point sets included).
  For collinear sets ``R`` is not unique, but ``S1_hat`` and ``err`` are.

The kernel (``csrc/procrustes.cu``) accumulates the moments in fp64 after shifting each row by its first selected
point, and finds ``R`` as the top eigenvector of Horn's 4x4 quaternion matrix of ``K``: the proper rotation maximising
``trace(R K)``, which is ``V Z U^T`` above.  ``oracle/procrustes_ref.py`` restates the rule with an SVD.
"""
import hashlib

import numpy as np
import torch

from . import _lib as L
from .misc import BodyPartIndices, shard_range


def average_pairwise_distance(joints3d, group=None):
    """APD = mean over ordered pairs (i != j) of mean-over-joints L2 distance (metric.py:8-37).

    Single-process by default, like the reference (which calls it on one rank only).  Sharding is OPT-IN: pass
    ``group=`` (a process group, or ``torch.distributed.group.WORLD``) and call it on EVERY rank of that group with
    the same ``joints3d``; each rank then reduces its contiguous row block and the partial sums are all-reduced."""
    L.require_cuda(joints3d, 'joints3d')
    j = joints3d.detach().to(torch.float32).contiguous()
    B, nj = j.shape[0], j.shape[1]
    world, rank = 1, 0
    if group is not None:
        import torch.distributed as dist
        world, rank = dist.get_world_size(group), dist.get_rank(group)
    row0, nrows = shard_range(B, world, rank)
    rows = torch.empty(max(nrows, 1), dtype=torch.float32, device=j.device)
    L.check(L.load().dpb_apd_partial(L.ptr(j), B, nj, row0, nrows, L.ptr(rows), L.current_stream(j.device)))
    out = rows[:nrows].double().sum().reshape(1)          # per-row fp32 sums, added in double
    if world > 1:
        dist.all_reduce(out, group=group)
    return (out / (B * (B - 1)))[0].float()


def mean_point_error_mm(a, b, idx=None):
    """Per-sample 1000 * mean_k ||a[:,k]-b[:,k]|| over an optional point subset (AMASS.py:286-296)."""
    L.require_cuda(a, 'a')
    a = a.detach().to(torch.float32).contiguous()
    b = b.detach().to(torch.float32).contiguous()
    B, n = a.shape[0], a.shape[1]
    out = torch.empty(B, dtype=torch.float32, device=a.device)
    ix = None if idx is None else torch.as_tensor(idx, dtype=torch.int32, device=a.device).contiguous()
    L.check(L.load().dpb_mean_point_error(L.ptr(a), L.ptr(b), B, n, L.ptr(ix), 0 if ix is None else ix.numel(),
                                          L.ptr(out), L.current_stream(a.device)))
    return out


class Evaler:
    """lib/dataset/AMASS.py:263-324 -- MPVPE / MPJPE per sample (mm), min over hypotheses.  With
    ``procrustes=True`` the results also hold ``pa_mpvpe_all`` and ``pa_mpjpe_body``: the same errors after similarity
    alignment (``reconstruction_error``) over the same point subsets, in mm."""

    def __init__(self, body_model, part=None, vert_idx=None, procrustes=False):
        self.body_model = body_model
        self.part = part
        self.procrustes = procrustes
        if part is not None:
            self.joint_idx = np.array(getattr(BodyPartIndices, part)) + 1     # skip pelvis
            self.vert_idx = None if vert_idx is None else np.asarray(vert_idx)
        else:
            self.joint_idx, self.vert_idx = None, None

    def eval_bodys(self, outs, gts):
        body_gt = self.body_model(pose_body=gts)
        body_out = self.body_model(pose_body=outs)
        res = {'mpvpe_all': mean_point_error_mm(body_out.v, body_gt.v, self.vert_idx).cpu().numpy(),
               'mpjpe_body': mean_point_error_mm(body_out.Jtr, body_gt.Jtr, self.joint_idx).cpu().numpy()}
        if self.procrustes:
            res['pa_mpvpe_all'] = (reconstruction_error(body_out.v, body_gt.v, None, self.vert_idx) * 1000).cpu().numpy()
            res['pa_mpjpe_body'] = (reconstruction_error(body_out.Jtr, body_gt.Jtr, None, self.joint_idx) * 1000) \
                .cpu().numpy()
        return res

    def multi_eval_bodys(self, outs, gts):
        res = [self.eval_bodys(outs[:, h], gts) for h in range(outs.shape[1])]
        return {k: np.min([r[k] for r in res], axis=0) for k in res[0]}


class MeshTopology:
    """Faces shared by a batch of meshes, uploaded once (``dpb_selfisect_create``).  ``faces`` [nF,3] integer, on any
    device; every id must lie in [0, n_vertices).  At most 32 768 faces (SMPL / SMPL-H: 13 776, SMPL-X: 20 908);
    more raise NotImplementedError."""

    def __init__(self, faces, n_vertices, device=None):
        import ctypes as C
        n_vertices = int(n_vertices)
        f = _host_faces(faces, n_vertices)
        self.n_faces, self.n_vertices = f.shape[0], n_vertices
        self.device = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        self._h = None
        h = C.c_void_p()
        L.check(L.load().dpb_selfisect_create(C.byref(h), f.ctypes.data_as(C.POINTER(C.c_int32)), self.n_faces,
                                              n_vertices, self.device.index or 0))
        self._h = h

    def __del__(self):
        if getattr(self, '_h', None) is not None and L._lib is not None:
            L._lib.dpb_selfisect_destroy(self._h)
            self._h = None

    def workspace_bytes(self, B):
        return int(L.load().dpb_selfisect_workspace_bytes(self._h, int(B)))

    def counts(self, vertices, selection=None, workspace=None):
        """Selected-face counts int32 [B] of vertices [B,V,3] (fp32, contiguous, on the handle's device; -1 for a mesh
        with a non-finite vertex), and the per-face selection written into ``selection`` (uint8 [B,nF]) when given.
        No host synchronisation, so the call can be captured in a CUDA graph (pass a preallocated ``workspace``)."""
        B = vertices.shape[0]
        out = torch.empty(B, dtype=torch.int32, device=vertices.device)
        if workspace is None:
            workspace = torch.empty(max(self.workspace_bytes(B), 1), dtype=torch.uint8, device=vertices.device)
        L.check(L.load().dpb_selfisect_run(self._h, L.ptr(vertices), B, L.ptr(out), L.ptr(selection),
                                            L.ptr(workspace), workspace.numel() * workspace.element_size(),
                                            L.current_stream(vertices.device)))
        return out


def _host_faces(faces, n_vertices):
    """faces as a contiguous int32 host array, after the shape, dtype and range checks (ValueError)."""
    f = faces.detach().cpu().numpy() if isinstance(faces, torch.Tensor) else np.asarray(faces)
    if not np.issubdtype(f.dtype, np.integer):
        raise ValueError(f'faces must be integer, got {f.dtype}')
    if f.ndim != 2 or f.shape[1] != 3 or f.shape[0] == 0:
        raise ValueError(f'faces must have shape [nF,3] with nF >= 1, got {tuple(f.shape)}')
    if f.min() < 0 or f.max() >= n_vertices:
        raise ValueError(f'face vertex ids must lie in [0, {n_vertices}), got [{f.min()}, {f.max()}]')
    return np.ascontiguousarray(f, dtype=np.int32)


_TOPOLOGIES = {}


def self_intersections_percentage(vertices, faces, return_selection=False):
    """SI of each mesh: 100 x (faces in at least one intersecting pair) / nF, the rule in this module's docstring.
    The reference's function (lib/utils/metric.py:41-89) keeps its name here; its body is not part of the checkout
    this was built from, so the call surface is this project's: one call scores a whole batch.

    vertices: [B,V,3] or [V,3] on CUDA (fp32 is used as is -- LBS output takes no copy; other floats are converted);
    faces: [nF,3] integer tensor or array on any device, or a ``MeshTopology``.  For a tensor or array the uploaded
    topology is cached per (face contents, V, device).
    Returns float32 percentages [B] (0-d for a single mesh) on the vertices' device, NaN for a mesh whose faces
    reference a non-finite vertex; with ``return_selection=True`` also the per-face selection, bool [B,nF] ([nF]).
    There is no CPU fallback: CPU vertices raise RuntimeError."""
    if not isinstance(vertices, torch.Tensor) or vertices.dim() not in (2, 3) or vertices.shape[-1] != 3 or \
            vertices.shape[-2] == 0 or (vertices.dim() == 3 and vertices.shape[0] == 0):
        raise ValueError(f'vertices must be a tensor of shape [B,V,3] or [V,3], got {getattr(vertices, "shape", None)}')
    single, V = vertices.dim() == 2, vertices.shape[-2]
    if isinstance(faces, MeshTopology):
        if faces.n_vertices != V:
            raise ValueError(f'topology was built for {faces.n_vertices} vertices, got {V}')
        topo = faces
        L.require_cuda(vertices, 'vertices')
    else:
        f = _host_faces(faces, V)
        L.require_cuda(vertices, 'vertices')
        key = (hashlib.sha1(f.tobytes()).hexdigest(), f.shape[0], V, str(vertices.device))
        topo = _TOPOLOGIES.get(key)
        if topo is None:
            topo = _TOPOLOGIES[key] = MeshTopology(f, V, vertices.device)
    v = vertices.detach()
    v = (v[None] if single else v).to(torch.float32).contiguous()
    sel = torch.empty(v.shape[0], topo.n_faces, dtype=torch.uint8, device=v.device) if return_selection else None
    cnt = topo.counts(v, sel)
    pct = torch.where(cnt < 0, torch.full(cnt.shape, float('nan'), dtype=torch.float64, device=cnt.device),
                      cnt.double() * 100.0 / topo.n_faces).float()
    if single:
        pct = pct[0]
        sel = None if sel is None else sel[0]
    return (pct, sel.bool()) if return_selection else pct


def _procrustes(S1, S2, idx, want_aligned, want_params):
    """Checks (ValueError before any library call; RuntimeError for CPU tensors), then one dpb_procrustes launch.
    Returns (single, err [B], aligned [B,n,3] or None, params [B,13] or None), fp32 on the inputs' device."""
    for name, x in (('S1', S1), ('S2', S2)):
        if not isinstance(x, torch.Tensor) or x.dim() not in (2, 3) or x.shape[-1] != 3 or x.shape[-2] == 0 or \
                (x.dim() == 3 and x.shape[0] == 0):
            raise ValueError(f'{name} must be a tensor of shape [B,n,3] or [n,3], got {getattr(x, "shape", None)}')
        if not x.is_floating_point():
            raise ValueError(f'{name} must be floating point, got {x.dtype}')
    if S1.shape != S2.shape:
        raise ValueError(f'S1 and S2 must have the same shape, got {tuple(S1.shape)} and {tuple(S2.shape)}')
    n = S1.shape[-2]
    ix = None
    if idx is not None:
        ix = np.asarray(idx.detach().cpu().numpy() if isinstance(idx, torch.Tensor) else idx)
        if ix.ndim != 1 or ix.size == 0 or not np.issubdtype(ix.dtype, np.integer):
            raise ValueError(f'idx must be a non-empty 1-D integer sequence, got {ix.dtype} {ix.shape}')
        if ix.min() < 0 or ix.max() >= n:
            raise ValueError(f'idx entries must lie in [0, {n}), got [{ix.min()}, {ix.max()}]')
    L.require_cuda(S1, 'S1')
    L.require_cuda(S2, 'S2')
    if S1.device != S2.device:
        raise ValueError(f'S1 and S2 must be on the same device, got {S1.device} and {S2.device}')
    single = S1.dim() == 2
    a = (S1.detach()[None] if single else S1.detach()).to(torch.float32).contiguous()
    b = (S2.detach()[None] if single else S2.detach()).to(torch.float32).contiguous()
    B = a.shape[0]
    if ix is not None:
        ix = torch.as_tensor(ix.astype(np.int32), device=a.device)
    err = torch.empty(B, dtype=torch.float32, device=a.device)
    aligned = torch.empty_like(a) if want_aligned else None
    params = torch.empty(B, 13, dtype=torch.float32, device=a.device) if want_params else None
    L.check(L.load().dpb_procrustes(L.ptr(a), L.ptr(b), B, n, L.ptr(ix), 0 if ix is None else ix.numel(), L.ptr(err),
                                    L.ptr(aligned), L.ptr(params), L.current_stream(a.device)))
    return single, err, aligned, params


def compute_similarity_transform(S1, S2, idx=None, return_params=False):
    """S1_hat: ``S1`` aligned to ``S2`` by the similarity transform of this module's docstring (reference
    lib/utils/transforms.py).  S1, S2: [B,n,3] or a single [n,3] pair, floating point, on CUDA (fp32 is used as is);
    ``idx``: optional host sequence of point ids that fit the transform (every point is still transformed).
    Returns fp32 S1_hat of S1's shape, and with ``return_params=True`` also ``(scale [B], R [B,3,3], t [B,3])``
    (without the batch dimension for a single pair).  NaN rows as in the docstring.  No host synchronisation unless
    ``idx`` is given (it is uploaded); there is no CPU fallback."""
    single, _, aligned, params = _procrustes(S1, S2, idx, True, return_params)
    if single:
        aligned = aligned[0]
    if not return_params:
        return aligned
    scale, R, t = params[:, 0], params[:, 1:10].reshape(-1, 3, 3), params[:, 10:]
    if single:
        scale, R, t = scale[0], R[0], t[0]
    return aligned, (scale, R, t)


def reconstruction_error(S1, S2, reduction='mean', idx=None):
    """PA-MPJPE / PA-MPVPE: the mean distance after similarity alignment, in the input's units (reference
    lib/utils/transforms.py).  Per row over the selected points ``idx`` (all when None); ``reduction`` 'mean' or 'sum'
    over rows gives a 0-d tensor, None the fp32 per-row errors [B] (0-d for a single [n,3] pair).  The row reduction
    runs on the device in fp64; with ``idx=None`` the call never synchronises with the host."""
    if reduction not in ('mean', 'sum', None):
        raise ValueError(f"reduction must be 'mean', 'sum' or None, got {reduction!r}")
    single, err, _, _ = _procrustes(S1, S2, idx, False, False)
    if reduction == 'mean':
        return err.double().mean().float()
    if reduction == 'sum':
        return err.double().sum().float()
    return err[0] if single else err
