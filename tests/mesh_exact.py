"""Exact distance and sign to a closed triangle mesh, in float64 numpy: the yardstick for the mesh signed distance.

Shares no code with the oracle (oracle/hp_oracle_mesh.h) or the kernels: the unsigned distance is Ericson's closest point
on a triangle (Real-Time Collision Detection, §5.1.5), minimised over all triangles; the sign comes from the generalized
winding number (sum of Van Oosterom-Strackee solid angles over 4 pi), which is +1 inside, 0 outside and needs no
pseudonormals, so it also handles nested shells and disjoint components. Inputs are the f32 vertices and query points
taken exactly, so the only error of the checker is float64 rounding (about 1e-16 of the coordinates)."""
import numpy as np

# nearest feature of the exact closest point
VERTEX, EDGE, FACE = 0, 1, 2
# Ericson's regions, in the order of his early exits: vertices A, B, edge AB, vertex C, edges AC, BC, face
_REGION_FEATURE = np.array([VERTEX, VERTEX, EDGE, VERTEX, EDGE, EDGE, FACE])


def _closest_on_triangles(p, A, B, C):
    """Closest points of points p (n, 3) on triangles (A, B, C) (m, 3) each: squared distance (n, m) and region (n, m)."""
    ab, ac = B - A, C - A
    ap = p[:, None, :] - A[None]
    bp = p[:, None, :] - B[None]
    cp = p[:, None, :] - C[None]
    d1, d2 = (ap * ab).sum(-1), (ap * ac).sum(-1)
    d3, d4 = (bp * ab).sum(-1), (bp * ac).sum(-1)
    d5, d6 = (cp * ab).sum(-1), (cp * ac).sum(-1)
    vc = d1 * d4 - d3 * d2
    vb = d5 * d2 - d1 * d6
    va = d3 * d6 - d5 * d4
    conds = [(d1 <= 0) & (d2 <= 0),
             (d3 >= 0) & (d4 <= d3),
             (vc <= 0) & (d1 >= 0) & (d3 <= 0),
             (d6 >= 0) & (d5 <= d6),
             (vb <= 0) & (d2 >= 0) & (d6 <= 0),
             (va <= 0) & (d4 - d3 >= 0) & (d5 - d6 >= 0)]
    region = np.select(conds, np.arange(6), 6)
    with np.errstate(divide="ignore", invalid="ignore"):
        denom = va + vb + vc
        t_bc = (d4 - d3) / ((d4 - d3) + (d5 - d6))
        # closest point = A + v ab + w ac
        v = np.select(conds, [0.0, 1.0, d1 / (d1 - d3), 0.0, 0.0, 1.0 - t_bc], vb / denom)
        w = np.select(conds, [0.0, 0.0, 0.0, 1.0, d2 / (d2 - d6), t_bc], vc / denom)
    r = ap - v[..., None] * ab[None] - w[..., None] * ac[None]
    return (r * r).sum(-1), region


def closest(verts, tris, pts, pair_budget=1 << 19):
    """Exact unsigned distance of every point to the mesh, with the triangle and the nearest feature (VERTEX / EDGE / FACE)
    of its closest point. Chunked over points and triangles so that 20 k x 20 k pairs take no more than a few hundred MB."""
    V = np.asarray(verts, np.float64)
    T = np.asarray(tris, np.int64)
    P = np.asarray(pts, np.float64)
    A, B, C = V[T[:, 0]], V[T[:, 1]], V[T[:, 2]]
    n, m = len(P), len(T)
    best = np.full(n, np.inf)
    tri = np.zeros(n, np.int64)
    region = np.zeros(n, np.int64)
    tchunk = max(1, min(m, pair_budget // 64))
    pchunk = max(1, pair_budget // tchunk)
    for i in range(0, n, pchunk):
        sl = slice(i, min(n, i + pchunk))
        for j in range(0, m, tchunk):
            d2, reg = _closest_on_triangles(P[sl], A[j:j + tchunk], B[j:j + tchunk], C[j:j + tchunk])
            k = d2.argmin(1)
            dk = d2[np.arange(len(k)), k]
            better = dk < best[sl]
            best[sl] = np.where(better, dk, best[sl])
            tri[sl] = np.where(better, j + k, tri[sl])
            region[sl] = np.where(better, reg[np.arange(len(k)), k], region[sl])
    return np.sqrt(best), tri, _REGION_FEATURE[region]


def winding_number(verts, tris, pts, pair_budget=1 << 19):
    """Generalized winding number of the mesh at every point: sum over triangles of the solid angle / (4 pi). For a closed,
    consistently outward-oriented mesh it is the number of shells around the point (1 inside, 0 outside, 0 in a cavity)."""
    V = np.asarray(verts, np.float64)
    T = np.asarray(tris, np.int64)
    P = np.asarray(pts, np.float64)
    A, B, C = V[T[:, 0]], V[T[:, 1]], V[T[:, 2]]
    out = np.zeros(len(P))
    tchunk = max(1, min(len(T), pair_budget // 64))
    pchunk = max(1, pair_budget // tchunk)
    for i in range(0, len(P), pchunk):
        p = P[i:i + pchunk, None, :]
        for j in range(0, len(T), tchunk):
            a, b, c = A[None, j:j + tchunk] - p, B[None, j:j + tchunk] - p, C[None, j:j + tchunk] - p
            la, lb, lc = (np.sqrt((x * x).sum(-1)) for x in (a, b, c))
            num = (a * np.cross(b, c)).sum(-1)
            den = la * lb * lc + (a * b).sum(-1) * lc + (b * c).sum(-1) * la + (c * a).sum(-1) * lb
            out[i:i + pchunk] += np.arctan2(num, den).sum(1)
    return out / (2 * np.pi)


def signed_distance(verts, tris, pts):
    """(signed exact distance, closest triangle, its nearest feature, winding number): the distance is negative where the
    winding number is above 1/2."""
    d, tri, feat = closest(verts, tris, pts)
    w = winding_number(verts, tris, pts)
    return np.where(w > 0.5, -d, d), tri, feat, w


def pseudonormals(verts, tris):
    """Float64 outward directions per feature, for placing points: unit face normals (nt, 3); per undirected edge the
    normalised sum of its two face normals (edges (ne, 2) sorted vertex pairs, normals (ne, 3)); per vertex the
    angle-weighted normal (nv, 3)."""
    V = np.asarray(verts, np.float64)
    T = np.asarray(tris, np.int64)
    A, B, C = V[T[:, 0]], V[T[:, 1]], V[T[:, 2]]
    fn = np.cross(B - A, C - A)
    fn /= np.linalg.norm(fn, axis=1, keepdims=True)
    e = np.sort(np.stack([T[:, [0, 1]], T[:, [1, 2]], T[:, [2, 0]]], 1).reshape(-1, 2), 1)
    edges, inv = np.unique(e, axis=0, return_inverse=True)
    en = np.zeros((len(edges), 3))
    np.add.at(en, inv.ravel(), np.repeat(fn, 3, 0))
    en /= np.linalg.norm(en, axis=1, keepdims=True)
    vn = np.zeros_like(V)
    for k in range(3):
        p0, p1, p2 = V[T[:, k]], V[T[:, (k + 1) % 3]], V[T[:, (k + 2) % 3]]
        u, w = p1 - p0, p2 - p0
        ang = np.arctan2(np.linalg.norm(np.cross(u, w), axis=1), (u * w).sum(1))
        np.add.at(vn, T[:, k], fn * ang[:, None])
    vn /= np.maximum(np.linalg.norm(vn, axis=1, keepdims=True), 1e-300)
    return fn, edges, en, vn
