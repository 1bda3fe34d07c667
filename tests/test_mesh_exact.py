"""CPU: the exact mesh checker (mesh_exact.py) against closed forms, the oracle's half-edge pairing rule, and the oracle's
mesh signed distance against exact geometry.

The oracle restates the reference bit for bit and the device copies the oracle bit for bit, so these tests are what ties
the three to the true distance. check_against_exact is shared with test_gpu_mesh_shapes.py, which applies it to the device."""
import numpy as np
import pytest

import meshgen
from mesh_exact import EDGE, FACE, VERTEX, closest, pseudonormals, signed_distance, winding_number

U = 2.0 ** -24                      # f32 unit roundoff

# |d - d_exact| <= K u (|p|inf + |v|inf) where the reference's EPS is below f32 resolution (meshgen.eps_reach <= 1e-7).
# With the region chosen right, the reference's d = |p - q| rounds each coordinate of the closest point q about three
# times (an edge vector or barycentric product, its scaling, the sum with a vertex) and p - q once, each rounding at most
# u (|p|inf + |v|inf); a coordinate error e gives at most sqrt(3) e in the 2-norm, so 4 sqrt(3) < 7, and the f32 dot
# product and square root add about 2u of |d|, itself below |p|inf + |v|inf, relative to that scale: K = 8. A region
# chosen wrong within f32 noise of its boundary moves q by the same order. Measured at most 2.2.
K = 8

# Second reference quirk, found by these tests: on sliver triangles the face branch of ClosestSimplexToPt computes the
# closest point from barycentrics u = va / (va + vb + vc) of unnormalised triple products, whose rounding error is about
# u * l_max^2 / (2 A) of the longest edge. For a point near the surface that in-plane error is the distance error. Only
# points whose exact closest feature is the face of a triangle with l_max^2 / (2 A) above SLIVER_ASPECT may exceed the
# bound, and they are counted per shape: at most SLIVER_EXCLUSIONS[shape] of them over all point classes.
SLIVER_ASPECT = 100.0
SLIVER_EXCLUSIONS = {"bipyramid_4096": 127}


def exact_shape(name):
    """(vertices, triangles, scale) of meshgen.SHAPES[name] where the reference's EPS is below f32 resolution: the small
    shapes scaled by EXACT_SCALE, the 4096-translated and the 1000-scaled cube as they are."""
    v, t = meshgen.SHAPES[name]()
    s = meshgen.EXACT_SCALE if meshgen.eps_reach(v, t) > 1e-7 else 1.0
    return meshgen.scaled((v, t), s) + (s,)


def aspect(v, t):
    V = v.astype(np.float64)
    A, B, C = V[t[:, 0]], V[t[:, 1]], V[t[:, 2]]
    lmax = np.max([np.linalg.norm(B - A, axis=1), np.linalg.norm(C - B, axis=1), np.linalg.norm(A - C, axis=1)], 0)
    return lmax ** 2 / np.linalg.norm(np.cross(B - A, C - A), axis=1)


def check_against_exact(name, v, t, sets, dist):
    """dist(points) -> f32 signed distances of the mesh (v, t) for every point class of `sets`; assert the K bound and the
    winding sign beyond it, outside the counted sliver exclusion. Returns {class: (worst error / bound unit, excluded)}."""
    assert meshgen.eps_reach(v, t) <= 1e-7, name
    asp = aspect(v, t)
    vmax = np.abs(v.astype(np.float64)).max()
    report, excluded = {}, 0
    for cls, p in sets.items():
        d = dist(p).astype(np.float64)
        ex, tri, feat, w = signed_distance(v, t, p)
        unit = U * (np.abs(p.astype(np.float64)).max(1) + vmax)
        err = np.abs(np.abs(d) - np.abs(ex)) / unit
        sliver = (feat == FACE) & (asp[tri] > SLIVER_ASPECT)
        over = err > K
        bad = np.flatnonzero(over & ~sliver)
        assert len(bad) == 0, "%s/%s: %d points off by more than %d u, first %s: d %r exact %r, feature %d of triangle %d" % (
            name, cls, len(bad), K, p[bad[0]].tolist(), d[bad[0]], ex[bad[0]], feat[bad[0]], tri[bad[0]])
        sep = np.abs(ex) > K * unit
        wrong = np.flatnonzero(sep & (np.sign(d) != np.sign(ex)) & ~(over & sliver))
        assert len(wrong) == 0, "%s/%s: %d points with the wrong sign, first %s: d %r exact %r winding %r feature %d" % (
            name, cls, len(wrong), p[wrong[0]].tolist(), d[wrong[0]], ex[wrong[0]], w[wrong[0]], feat[wrong[0]])
        excluded += int((over & sliver).sum())
        report[cls] = (float(err[~(over & sliver)].max()), int((over & sliver).sum()))
    assert excluded <= SLIVER_EXCLUSIONS.get(name, 0), (name, excluded)
    return report


def format_report(report):
    return " ".join("%s %.2f%s" % (c, e, "/%d excl" % x if x else "") for c, (e, x) in report.items())


# ---- the checker against closed forms ---------------------------------------------------------------------------------------
def box_sdf(p, h):
    q = np.abs(p) - h
    return np.linalg.norm(np.maximum(q, 0), axis=1) + np.minimum(q.max(1), 0)


def octahedron_sdf(p, s):
    """Exact distance to the solid |x| + |y| + |z| <= s (the closed form of I. Quilez's 'distance functions' page)."""
    p = np.abs(p)
    m = p.sum(1) - s
    out = m / np.sqrt(3.0)
    for axis in range(3):
        q = np.roll(p, -axis, 1)                               # q = p.xyz, p.yzx, p.zxy
        take = (3 * p[:, axis] < m) & ~np.any([3 * p[:, a] < m for a in range(axis)], 0) if axis else 3 * p[:, 0] < m
        k = np.clip(0.5 * (q[:, 2] - q[:, 1] + s), 0.0, s)
        r = np.linalg.norm(np.stack([q[:, 0], q[:, 1] - s + k, q[:, 2] - k], 1), axis=1)
        out = np.where(take, r, out)
    return out


def test_checker_matches_closed_form_box_and_octahedron():
    rng = np.random.default_rng(0)
    for k in (1, 3):
        v, t = meshgen.box_mesh(k, 0.3)
        h = float(v.max())
        c = rng.choice([-h, h], (3000, 3))
        c[:1000, 0] = rng.uniform(-h, h, 1000)                  # edges, then corners
        p = np.concatenate([rng.uniform(-2 * h, 2 * h, (3000, 3)), c + rng.normal(0, 1, (3000, 3)) * h * 10.0 ** rng.uniform(-6, -1, (3000, 1))])
        sd, _, _, w = signed_distance(v, t, p)
        assert np.abs(sd - box_sdf(p, h)).max() <= 1e-12
    v, t = meshgen.octahedron(0.3)
    s = float(v.max())
    p = np.concatenate([rng.uniform(-2 * s, 2 * s, (4000, 3)), v[rng.integers(0, 6, 2000)] + rng.normal(0, 1e-3, (2000, 3))])
    sd, _, _, _ = signed_distance(v, t, p)
    assert np.abs(sd - octahedron_sdf(p, s)).max() <= 1e-12


def test_winding_number_counts_shells():
    rng = np.random.default_rng(1)
    d = rng.normal(size=(3000, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    v, t = meshgen.hollow_ball(0.3, 0.2)                    # inscribed radii above 0.28 and 0.18
    r = np.concatenate([rng.uniform(0, 0.15, 1000), rng.uniform(0.22, 0.27, 1000), rng.uniform(0.32, 3.0, 1000)])
    w = winding_number(v, t, d * r[:, None])
    assert np.abs(w - np.repeat([0.0, 1.0, 0.0], 1000)).max() <= 1e-9
    v, t = meshgen.tetrahedra_sharing_vertex()
    cen = np.stack([v[t[:4]].mean((0, 1)), v[t[4:]].mean((0, 1)), v[0] * 3.0])
    assert np.abs(winding_number(v, t, cen) - [1.0, 1.0, 0.0]).max() <= 1e-9


def test_nearest_feature_classification():
    v, t = meshgen.box_mesh(2, 0.3)
    fn, edges, en, vn = pseudonormals(v, t)
    V = v.astype(np.float64)
    corners = np.flatnonzero((np.abs(V) == V.max()).all(1))
    sharp = np.flatnonzero((np.abs(V[edges]) == V.max()).sum(2).min(1) >= 2)
    for delta in (1e-6, 1e-2):
        _, _, f = closest(v, t, V[corners] + delta * vn[corners])
        assert (f == VERTEX).all()
        _, _, f = closest(v, t, V[edges[sharp]].mean(1) + delta * en[sharp])
        assert (f == EDGE).all()
        _, _, f = closest(v, t, V[t].mean(1) + delta * fn)
        assert (f == FACE).all()


# ---- half-edge pairing -----------------------------------------------------------------------------------------------------
def map_pairing(tris):
    """Mesh::CreateHalfEdges's std::map sequence in half-edge order: pair with the stored reverse edge if there is one, else
    store this edge unless the same direction is already stored. None if a half-edge stays unpaired."""
    flat = np.asarray(tris, np.int64).reshape(-1)
    he = np.full(len(flat), 0xFFFFFFFF, np.uint32)
    known = {}
    for i, a in enumerate(flat):
        b = flat[i - 2] if i % 3 == 2 else flat[i + 1]
        j = known.get((b, a))
        if j is not None and j != i:
            he[i], he[j] = j, i
        elif (a, b) not in known:
            known[(a, b)] = i
    return None if (he == 0xFFFFFFFF).any() else he


def oriented_tet(v, ids):
    """The 4 outward triangles of the tetrahedron on vertices ids of v."""
    out = []
    for k in range(4):
        f = [ids[j] for j in range(4) if j != k]
        a, b, c = v[f].astype(np.float64)
        if np.dot(np.cross(b - a, c - a), a - v[ids[k]]) < 0:
            f = [f[0], f[2], f[1]]
        out.append(f)
    return out


def pairing_meshes():
    """name -> (vertices, triangles, accepted)."""
    v1, t1 = meshgen.tetrahedron(0.3)
    v2 = np.concatenate([v1, -v1[2:]]).astype(np.float32)                       # a second tetrahedron on the edge (0, 1)
    t2 = np.concatenate([t1, oriented_tet(v2, [0, 1, 4, 5])]).astype(np.uint32)
    v3 = np.concatenate([v1, [[0.9, 0.9, 0.9], [0.95, 0.9, 0.9]]]).astype(np.float32)
    t3 = np.concatenate([t1, [[4, 4, 5]]]).astype(np.uint32)
    flipped = t1.copy()
    flipped[2] = flipped[2, ::-1]
    out = dict(tetrahedra_sharing_edge=(v2, t2, False), degenerate_triangle=(v3, t3, False),
               flipped_triangle=(v1, flipped, False), tetrahedron=(v1, t1, True))
    for name in ("tetrahedra_sharing_vertex", "cube_k3", "octahedron", "star_prism", "bipyramid_3", "hollow_ball", "torus"):
        v, t = meshgen.SHAPES[name]()
        out[name] = (v, t, True)
    return out


def test_pairing_rule_accepts_rejects_and_pins_twins(oracle):
    for name, (v, t, accepted) in pairing_meshes().items():
        want = map_pairing(t)
        assert (want is not None) == accepted, name
        if not accepted:
            with pytest.raises(ValueError):
                oracle.OracleMesh(v, t)
            continue
        om = oracle.OracleMesh(v, t)
        assert np.array_equal(om.half_edges(), want), name
        om.close()


def test_reference_mesh_agrees_on_pairing(ref):
    for name, (v, t, accepted) in pairing_meshes().items():
        assert (ref.RefMesh.create(v, t) is not None) == accepted, name


# ---- the oracle against exact geometry ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(meshgen.SHAPES))
def test_oracle_distance_matches_exact_geometry(oracle, name):
    v, t, s = exact_shape(name)
    om = oracle.OracleMesh(v, t)
    sets = meshgen.point_sets(v, t, np.random.default_rng(sum(map(ord, name))))
    report = check_against_exact(name, v, t, sets, lambda p: om.sdf(p, True, 8))
    print("%s (%d triangles, x%g): worst |d - exact| / u(|p| + |v|) per class: %s" % (
        name, len(t), s, format_report(report)))


def test_torus_deviation_from_exact_geometry(oracle):
    """The 60 x 40 torus at its own scale, where the reference's EPS reaches about 0.02 from an edge line: print how far the
    reference's distance is from the exact one, on the golden points and on points hugging the surface."""
    from common import golden
    v, t = meshgen.bumpy_torus(60, 40)
    om = oracle.OracleMesh(v, t)
    g = golden("mesh_torus")
    V = v.astype(np.float64)
    rng = np.random.default_rng(2)
    cen = V[t[rng.integers(0, len(t), 2000)]].mean(1)
    near = (cen + rng.normal(0, 1, cen.shape) * 10.0 ** rng.uniform(-4, -2, (2000, 1))).astype(np.float32)
    for label, p in (("golden points", g["pts"][:4000]), ("points 1e-4..1e-2 from the surface", near)):
        d = om.sdf(p, True, 8).astype(np.float64)
        ex, _, feat, _ = signed_distance(v, t, p)
        err = np.abs(np.abs(d) - np.abs(ex))
        wrong = (np.sign(d) != np.sign(ex)) & (np.abs(ex) > 1e-4)
        print("torus 60x40, %d %s: |d - exact| median %.2g, > 1e-5: %d, > 1e-3: %d, max %.2g; wrong sign beyond 1e-4: %d" % (
            len(p), label, np.median(err), (err > 1e-5).sum(), (err > 1e-3).sum(), err.max(), wrong.sum()))
        assert meshgen.eps_reach(v, t) > 1e-7                  # the reason: EPS is far above f32 resolution here
