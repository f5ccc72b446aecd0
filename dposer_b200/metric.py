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
    """lib/dataset/AMASS.py:263-324 -- MPVPE / MPJPE per sample (mm), min over hypotheses."""

    def __init__(self, body_model, part=None, vert_idx=None):
        self.body_model = body_model
        self.part = part
        if part is not None:
            self.joint_idx = np.array(getattr(BodyPartIndices, part)) + 1     # skip pelvis
            self.vert_idx = None if vert_idx is None else np.asarray(vert_idx)
        else:
            self.joint_idx, self.vert_idx = None, None

    def eval_bodys(self, outs, gts):
        body_gt = self.body_model(pose_body=gts)
        body_out = self.body_model(pose_body=outs)
        return {'mpvpe_all': mean_point_error_mm(body_out.v, body_gt.v, self.vert_idx).cpu().numpy(),
                'mpjpe_body': mean_point_error_mm(body_out.Jtr, body_gt.Jtr, self.joint_idx).cpu().numpy()}

    def multi_eval_bodys(self, outs, gts):
        res = [self.eval_bodys(outs[:, h], gts) for h in range(outs.shape[1])]
        return {k: np.min([r[k] for r in res], axis=0) for k in ('mpvpe_all', 'mpjpe_body')}


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
