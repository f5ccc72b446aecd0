"""Self-intersection metric (SI, reference ``self_intersections_percentage`` lib/utils/metric.py:41-89) as a float64
numpy restatement of the specification in ``dposer_b200.metric`` -- TEST INFRASTRUCTURE ONLY.

The reference computes SI with pymeshlab (VCG ``Clean::SelfIntersections``); neither is available here, so parity
with pymeshlab is unpinned.  This module and ``csrc/selfisect.cu`` evaluate the same fp64 formulas on the fp32
inputs, operation for operation (no fused multiply-adds, the same association), so their per-face selections are
compared for equality.

Broad phase: sweep-and-prune of the face AABBs along the axis of largest extent, then the exact closed AABB overlap
test on all three axes.  It is complete: two closed triangles with a common point have overlapping AABBs.
"""
import numpy as np


def _cross(a, b):
    return np.stack([a[:, 1] * b[:, 2] - a[:, 2] * b[:, 1],
                     a[:, 2] * b[:, 0] - a[:, 0] * b[:, 2],
                     a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0]], axis=1)


def _dot(a, b):
    return a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1] + a[:, 2] * b[:, 2]


def _orient(n, p, q, r):
    """Orientation of (p, q, r) in the plane with normal n: sign of n . ((q - p) x (r - p))."""
    return _dot(n, _cross(q - p, r - p))


def _on_segment(p, c, e):
    """p (collinear with c, e) lies on the closed segment [c, e]."""
    return (_dot(p - c, e - c) >= 0) & (_dot(p - e, c - e) >= 0)


def _segments_meet(n, a, b, c, e):
    """Closed coplanar segments [a, b] and [c, e] have a common point."""
    d1, d2 = _orient(n, c, e, a), _orient(n, c, e, b)
    d3, d4 = _orient(n, a, b, c), _orient(n, a, b, e)
    proper = (((d1 > 0) & (d2 < 0)) | ((d1 < 0) & (d2 > 0))) & (((d3 > 0) & (d4 < 0)) | ((d3 < 0) & (d4 > 0)))
    touch = (((d1 == 0) & _on_segment(a, c, e)) | ((d2 == 0) & _on_segment(b, c, e)) |
             ((d3 == 0) & _on_segment(c, a, b)) | ((d4 == 0) & _on_segment(e, a, b)))
    return proper | touch


def _inside(n, p, q0, q1, q2):
    return (_orient(n, q0, q1, p) >= 0) & (_orient(n, q1, q2, p) >= 0) & (_orient(n, q2, q0, p) >= 0)


def _volumes(a, b, q0, q1, q2):
    """Signed volumes proportional to the barycentric coordinates where line a->b crosses plane (q0, q1, q2)."""
    d = b - a
    return (_dot(d, _cross(q1 - a, q2 - a)), _dot(d, _cross(q2 - a, q0 - a)), _dot(d, _cross(q0 - a, q1 - a)))


def segment_meets_triangle(a, b, q0, q1, q2, n):
    """Closed segment [a, b] and closed triangle (q0, q1, q2) with normal n = (q1 - q0) x (q2 - q0) != 0."""
    da, db = _dot(n, a - q0), _dot(n, b - q0)
    same = ((da > 0) & (db > 0)) | ((da < 0) & (db < 0))
    coplanar = (da == 0) & (db == 0)
    v0, v1, v2 = _volumes(a, b, q0, q1, q2)
    hit3 = ((v0 >= 0) & (v1 >= 0) & (v2 >= 0)) | ((v0 <= 0) & (v1 <= 0) & (v2 <= 0))
    hit2 = (_inside(n, a, q0, q1, q2) | _inside(n, b, q0, q1, q2) | _segments_meet(n, a, b, q0, q1) |
            _segments_meet(n, a, b, q1, q2) | _segments_meet(n, a, b, q2, q0))
    return ~same & np.where(coplanar, hit2, hit3)


def segment_pierces_interior(a, b, q0, q1, q2, n):
    """a and b strictly on opposite sides of the plane, crossing point strictly inside the triangle."""
    da, db = _dot(n, a - q0), _dot(n, b - q0)
    opposite = ((da > 0) & (db < 0)) | ((da < 0) & (db > 0))
    v0, v1, v2 = _volumes(a, b, q0, q1, q2)
    return opposite & (((v0 > 0) & (v1 > 0) & (v2 > 0)) | ((v0 < 0) & (v1 < 0) & (v2 < 0)))


def _halfway_test(P, Ff, Fg, i, ng):
    """s = 1: the edge of f opposite its shared vertex Ff[i], moved halfway to it, pierces g's interior."""
    k = np.arange(len(i))
    v = P[Ff[k, i]]
    m1 = (v + P[Ff[k, (i + 1) % 3]]) * 0.5
    m2 = (v + P[Ff[k, (i + 2) % 3]]) * 0.5
    return segment_pierces_interior(m1, m2, P[Fg[:, 0]], P[Fg[:, 1]], P[Fg[:, 2]], ng)


def pairs_intersect(P, F, f, g, normals):
    """Decision of the specification for face pairs (f[k], g[k]), f != g, both of non-zero area."""
    Ff, Fg = F[f], F[g]
    eq = Ff[:, :, None] == Fg[:, None, :]                     # [N, 3 (f), 3 (g)]
    in_g = eq.any(2)
    s = in_g.sum(1)
    out = s == 3
    m0 = np.nonzero(s == 0)[0]
    if len(m0):
        a = [P[Ff[m0, j]] for j in range(3)]
        b = [P[Fg[m0, j]] for j in range(3)]
        nf, ng = normals[f[m0]], normals[g[m0]]
        hit = np.zeros(len(m0), bool)
        for j in range(3):
            hit |= segment_meets_triangle(a[j], a[(j + 1) % 3], b[0], b[1], b[2], ng)
        for j in range(3):
            hit |= segment_meets_triangle(b[j], b[(j + 1) % 3], a[0], a[1], a[2], nf)
        out[m0] = hit
    m1 = np.nonzero(s == 1)[0]
    if len(m1):
        i = np.argmax(in_g[m1], axis=1)
        j = np.argmax(eq[m1].any(1), axis=1)
        out[m1] = (_halfway_test(P, Ff[m1], Fg[m1], i, normals[g[m1]]) |
                   _halfway_test(P, Fg[m1], Ff[m1], j, normals[f[m1]]))
    return out


def face_normals(P, F):
    p0, p1, p2 = P[F[:, 0]], P[F[:, 1]], P[F[:, 2]]
    return _cross(p1 - p0, p2 - p0)


def candidate_pairs(P32, F, valid, chunk=1 << 22):
    """All pairs (f < g) of valid faces whose closed fp32 AABBs overlap (sweep-and-prune, complete)."""
    tri = P32[F]                                              # [nF, 3, 3] fp32
    lo, hi = tri.min(1), tri.max(1)
    idx = np.nonzero(valid)[0]
    if len(idx) < 2:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    lo_v, hi_v = lo[idx], hi[idx]
    ax = int(np.argmax(hi_v.max(0).astype(np.float64) - lo_v.min(0)))
    order = np.argsort(lo_v[:, ax], kind='stable')
    los = lo_v[order, ax]
    end = np.searchsorted(los, hi_v[order, ax], side='right')
    cnt = np.maximum(end - np.arange(len(order)) - 1, 0)
    fs, gs = [], []
    starts = np.concatenate([[0], np.cumsum(cnt)])
    a0 = 0
    while a0 < len(order):                                    # bounded memory: blocks of about `chunk` pairs
        a1 = int(np.searchsorted(starts, starts[a0] + chunk, side='right'))
        a1 = min(max(a1 - 1, a0 + 1), len(order))
        c = cnt[a0:a1]
        ia = np.repeat(np.arange(a0, a1), c)
        ib = ia + 1 + (np.arange(c.sum()) - np.repeat(starts[a0:a1] - starts[a0], c))
        ff, gg = idx[order[ia]], idx[order[ib]]
        ok = np.all((lo[ff] <= hi[gg]) & (lo[gg] <= hi[ff]), axis=1)
        ff, gg = ff[ok], gg[ok]
        fs.append(np.minimum(ff, gg))
        gs.append(np.maximum(ff, gg))
        a0 = a1
    return np.concatenate(fs), np.concatenate(gs)


def selection(vertices, faces, pairs=None):
    """Per-face selection (bool [nF]) and SI in percent (NaN when a face references a non-finite vertex).
    pairs: optional (f, g) candidate arrays replacing the broad phase (the brute-force check passes all pairs)."""
    P32 = np.ascontiguousarray(np.asarray(vertices, dtype=np.float32))
    F = np.ascontiguousarray(np.asarray(faces, dtype=np.int64))
    nF = F.shape[0]
    sel = np.zeros(nF, bool)
    if not np.isfinite(P32[F]).all():
        return sel, float('nan')
    P = P32.astype(np.float64)
    normals = face_normals(P, F)
    valid = np.any(normals != 0, axis=1)
    if pairs is None:
        f, g = candidate_pairs(P32, F, valid)
    else:
        f, g = (np.asarray(x, np.int64) for x in pairs)
        tri = P32[F]
        lo, hi = tri.min(1), tri.max(1)
        keep = (f != g) & valid[f] & valid[g] & np.all((lo[f] <= hi[g]) & (lo[g] <= hi[f]), axis=1)
        f, g = np.minimum(f, g)[keep], np.maximum(f, g)[keep]
    hit = pairs_intersect(P, F, f, g, normals) if len(f) else np.zeros(0, bool)
    sel[f[hit]] = True
    sel[g[hit]] = True
    return sel, 100.0 * sel.sum() / nF


def brute_force_selection(vertices, faces):
    """The same decision on every pair of faces (O(nF^2)), for small meshes."""
    nF = len(faces)
    f, g = np.triu_indices(nF, 1)
    return selection(vertices, faces, pairs=(f, g))


def explain(vertices, faces, face):
    """Debug report for one face: every AABB-overlapping partner g with (g, shared vertex count, decision, smallest
    |plane-side determinant| n . (x - q0) over the vertices of both faces), to judge how close a decision was."""
    P32 = np.asarray(vertices, np.float32)
    F = np.asarray(faces, np.int64)
    P = P32.astype(np.float64)
    normals = face_normals(P, F)
    tri = P32[F]
    lo, hi = tri.min(1), tri.max(1)
    g = np.nonzero(np.all((lo <= hi[face]) & (lo[face] <= hi), axis=1) & np.any(normals != 0, axis=1))[0]
    g = g[g != face]
    f = np.full_like(g, face)
    hit = pairs_intersect(P, F, f, g, normals)
    rows = []
    for k, gg in enumerate(g):
        s = len(set(F[face]) & set(F[gg]))
        d = [abs(float(normals[gg] @ (P[v] - P[F[gg, 0]]))) for v in F[face]]
        d += [abs(float(normals[face] @ (P[v] - P[F[face, 0]]))) for v in F[gg]]
        rows.append((int(gg), s, bool(hit[k]), min(x for x in d if x > 0) if any(x > 0 for x in d) else 0.0))
    return rows


def _two_faces(f, g, shared=()):
    """Mesh of triangles f and g (3x3 coordinates each); `shared` lists (i, j): g's vertex j IS f's vertex i."""
    P, Fg = [list(p) for p in f], []
    smap = dict((j, i) for i, j in shared)
    for j, q in enumerate(g):
        if j in smap:
            Fg.append(smap[j])
        else:
            Fg.append(len(P))
            P.append(list(q))
    return np.array(P, np.float32), np.array([[0, 1, 2], Fg], np.int32)


_F = [(0, 0, 0), (4, 0, 0), (0, 4, 0)]


def hand_cases():
    """name -> (vertices fp32 [V,3], faces int32 [2,3], expected selection bool [2], or None for SI = NaN).
    Small-integer coordinates: every fp64 expression is exact, so the outcomes are the geometric truth."""
    both, none = np.array([True, True]), np.array([False, False])
    c = {
        'crossing': (*_two_faces(_F, [(1, 1, -1), (1, 1, 1), (1, 5, 0)]), both),
        'disjoint': (*_two_faces(_F, [(1, 1, 1), (1, 1, 3), (1, 5, 2)]), none),
        'touch_vertex': (*_two_faces(_F, [(4, 0, 0), (6, 0, 1), (6, 1, 0)]), both),
        'touch_edge': (*_two_faces(_F, [(1, 0, 0), (3, 0, 0), (2, -2, 2)]), both),
        'coplanar_overlap': (*_two_faces(_F, [(1, 1, 0), (5, 1, 0), (1, 5, 0)]), both),
        'coplanar_disjoint': (*_two_faces(_F, [(5, 5, 0), (8, 5, 0), (5, 8, 0)]), none),
        's1_piercing': (*_two_faces(_F, [(0, 0, 0), (2, 2, 2), (2, 2, -2)], shared=[(0, 0)]), both),
        's1_not_piercing': (*_two_faces(_F, [(0, 0, 0), (2, 2, 2), (2, 2, 4)], shared=[(0, 0)]), none),
        's2_fold': (*_two_faces(_F, [(0, 0, 0), (4, 0, 0), (1, 1, 0)], shared=[(0, 0), (1, 1)]), none),
        'duplicate_face': (np.array(_F, np.float32), np.array([[0, 1, 2], [1, 2, 0]], np.int32), both),
        'zero_area': (*_two_faces(_F, [(1, 1, -1), (1, 1, 1), (1, 1, 3)]), none),
    }
    P, F = _two_faces(_F, [(1, 1, -1), (1, 1, 1), (1, 5, 0)])
    P[4, 2] = np.nan
    c['nan_vertex'] = (P, F, None)
    P2 = np.concatenate([P, [[np.nan, 0, 0]]]).astype(np.float32)
    P2[4, 2] = 1
    c['nan_unreferenced'] = (P2, F, both)
    return c
