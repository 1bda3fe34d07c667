"""hpsdf_query_bounds / Octree.QueryBounds: certified bounds of Query over axis-aligned boxes (DESIGN §14). Checked against
Query on dense samples of every box, against the independent checker (bounds_ref.py), against the exact sphere, and for the
structure the contract pins: nesting, covering boxes, point boxes, determinism across entry points, chunks and reruns."""
import os
import re
import subprocess

import numpy as np
import pytest
import scipy.optimize

import bounds_ref as B
from cases import CASES
from common import product_cfg
from test_gpu_derivatives import every_degree_block

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "hp-adaptive-signed-distance-field-octree_b200")
GXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
U = 2.0 ** -53


# ---- CPU: the checker on its own polynomials; the entry points without a device ----------------------------------------------

def one_leaf(degree, depth, seed):
    """A checker leaf of cell 1 on every axis at `depth` (interior, not on the root's boundary) with seeded coefficients."""
    rng = np.random.default_rng(seed)
    c = rng.normal(size=B.COUNTS[degree]) * 0.6 ** np.arange(B.COUNTS[degree]) ** 0.5
    return B.Leaves([[1, 1, 1]], [depth], [degree], [c])


def test_kappa_table_matches_its_derivation():
    src = open(os.path.join(PKG, "csrc", "bounds_kernels.cuh")).read()
    table = [int(x) for x in re.search(r"kBoundsKappaLog2\[kMaxDegree \+ 1\] = \{([^}]*)\}", src).group(1).split(",")]
    assert table == [B.kappa_log2(p) for p in range(13)]
    norms = [float(B.collocation_norm(p)) for p in range(1, 7)]
    assert np.allclose(norms, [1, 3, 5, 11.6667, 21, 46.2], rtol=1e-3) and 2.8e3 < float(B.collocation_norm(12)) < 3e3


def test_legendre_recurrence_error_is_inside_the_stated_bound():
    """Query's P_j by the three-term recurrence in f64 against mpmath: |error| <= 12 j^2 2^-53 for |u| <= 1 + 2^-14."""
    import mpmath as mp
    u = np.concatenate([np.linspace(-1 - 2.0 ** -14, 1 + 2.0 ** -14, 801), np.random.default_rng(1).uniform(-1, 1, 200)])
    rec = [((2 * j - 1) / j, (j - 1) / j) for j in range(1, 13)]
    for x in u:
        m2, m1 = 0.0, 1.0
        for j in range(1, 13):
            v = rec[j - 1][0] * x * m1 - rec[j - 1][1] * m2
            m2, m1 = m1, v
            assert abs(v - float(mp.legendre(j, mp.mpf(x)))) <= 12 * j * j * U


@pytest.mark.parametrize("degree", range(13))
def test_checker_hull_contains_its_polynomial(degree):
    rng = np.random.default_rng(degree)
    for depth in (0, 4, 10):
        lf = one_leaf(degree, depth, degree + 17 * depth)
        for _ in range(2):
            a, b = np.sort(rng.uniform(lf.elo[0], lf.ehi[0], (2, 3)), 0)
            (lo, hi), al = lf.interval(0, a, b)
            p = rng.uniform(a, b, (3000, 3))
            v = B.leaf_poly(lf.coeffs[0], degree, depth, (p - lf.c[0]) * 2.0 ** (depth + 1))
            slack = 1e-13 * float(lf.s[0])
            assert (v >= lo - slack).all() and (v <= hi + slack).all(), (degree, depth)
            assert hi - lo <= (v.max() - v.min()) * 4 + 4 * al + slack


def test_checker_hull_shrinks_quadratically():
    """The Bernstein coefficients of a sub-box approach the polynomial at their Greville points (k / p per axis) as O(h^2):
    the distance falls by about 4 each time the box halves, so the hull converges to the range quadratically."""
    for degree in (2, 4, 7):
        lf = one_leaf(degree, 3, 5 + degree)
        x0 = lf.c[0] + 0.013
        g = np.arange(degree + 1) / degree
        grev = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
        dist = []
        for k in range(5):
            h = 2.0 ** -(k + 6)
            _, _, bern = lf.hull(0, x0 - h, x0 + h)
            v = B.leaf_poly(lf.coeffs[0], degree, 3, (x0 - h + 2 * h * grev - lf.c[0]) * 16.0)
            dist.append(np.abs(bern.astype(np.float64).reshape(-1) - v).max())
        ratio = np.array(dist[:-1]) / np.array(dist[1:])
        assert (ratio > 3.5).all() and abs(ratio[-1] - 4.0) < 0.2, (degree, ratio)


def analytic_leaves(kind, depth=2):
    """A complete grid of leaves whose polynomials are the sphere |p|^2 - 0.3^2 (degree 2) or a plane (degree 1), as in
    test_gpu_raycast's checker tests; Legendre coefficients by a least-squares fit, exact up to rounding."""
    from numpy.polynomial import legendre as Lg
    deg = 2 if kind == "sphere" else 1
    nrm = np.array([0.3, -0.5, 0.81]) / np.linalg.norm([0.3, -0.5, 0.81])
    f = (lambda p: (p * p).sum(1) - 0.09) if kind == "sphere" else (lambda p: p @ nrm - 0.05)
    k = 2 ** depth
    cells = np.stack(np.meshgrid(*[np.arange(k)] * 3, indexing="ij"), -1).reshape(-1, 3)
    bi = B.basis_index(deg)
    g = np.cos(np.pi * (np.arange(deg + 2) + 0.5) / (deg + 2))
    u = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    nl = np.sqrt((2.0 * np.arange(deg + 1) + 1) * 2.0 ** depth)
    basis = np.stack([Lg.legval(u[:, 0], np.eye(deg + 1)[a]) * Lg.legval(u[:, 1], np.eye(deg + 1)[b]) * Lg.legval(u[:, 2], np.eye(deg + 1)[c])
                      * nl[a] * nl[b] * nl[c] for a, b, c in bi], 1)
    co = []
    for cell in cells:
        centre = (cell + 0.5) / k - 0.5
        co.append(np.linalg.lstsq(basis, f(centre + u / (2 * k)), rcond=None)[0])
    return B.Leaves(cells, [depth] * len(cells), [deg] * len(cells), co), f, nrm


@pytest.mark.parametrize("kind", ["sphere", "plane"])
def test_checker_reproduces_closed_form_ranges(kind):
    lv, f, nrm = analytic_leaves(kind)
    rng = np.random.default_rng(4)
    for _ in range(25):
        lo = rng.uniform(-0.5, 0.45, 3)
        hi = np.minimum(lo + rng.uniform(0.0, 0.5, 3) ** 2, 0.5)
        f_lo, f_hi, tl, th = lv.bounds(lo, hi)
        if kind == "sphere":
            near = np.clip(0.0, lo, hi)
            far = np.where(np.abs(lo) > np.abs(hi), lo, hi)
            want = ((near ** 2).sum() - 0.09, (far ** 2).sum() - 0.09)
        else:
            want = (nrm @ np.where(nrm > 0, lo, hi) - 0.05, nrm @ np.where(nrm > 0, hi, lo) - 0.05)
        # a degree-2 hull is not the range on sub-boxes that straddle a leaf's extremum, so the sphere is exact at the
        # box's extremes only when they are attained at Bernstein vertices: there the hull equals the range
        assert f_lo <= want[0] + 1e-12 and f_hi >= want[1] - 1e-12
        if kind == "plane":
            assert abs(f_lo - want[0]) <= tl + 1e-12 and abs(f_hi - want[1]) <= th + 1e-12
        else:
            assert f_hi - want[1] <= th + 1e-12


def test_bounds_without_a_gpu_fail_with_no_device(hp):
    if hp.device_count() > 0:
        pytest.skip("a GPU is present")
    L = hp.lib()
    x, v = np.zeros((2, 3)), np.empty(2)
    assert L.hpsdf_query_bounds(None, x.ctypes.data, x.ctypes.data, 2, v.ctypes.data, v.ctypes.data) == hp.ERR_NO_DEVICE
    assert L.hpsdf_query_bounds_device(None, 0, 0, 0, 0, 0, None) == hp.ERR_NO_DEVICE
    for call in (lambda: hp.Octree().QueryBounds(np.zeros((2, 3)), np.ones((2, 3))), lambda: hp.Octree().QueryBoundsDevice(0, 0, 0, 0, 0)):
        with pytest.raises(hp.HpsdfError) as e:
            call()
        assert e.value.status == hp.ERR_NO_DEVICE


# ---- GPU: trees and boxes ------------------------------------------------------------------------------------------------------

TREES = ["csg_small", "c2_csg", "sphere_poly_1e8", "custom_domain", "mesh_torus", "every_degree"]


@pytest.fixture(scope="module")
def trees(hp):
    out = {}
    for name in ("csg_small", "c2_csg", "sphere_poly_1e8", "custom_domain"):
        cfg, prog = product_cfg(hp, name)
        t = hp.Octree()
        t.Create(cfg, prog)
        out[name] = t
    from meshgen import bumpy_torus, mesh_root
    v, tr = bumpy_torus(80, 40)
    lo, hi = mesh_root(v)
    t = hp.Octree()
    t.Create(hp.Config(target_error_threshold=1e-6, continuity_enforce=0, root_min=lo, root_max=hi), hp.SdfProgram([("mesh", [], hp.Mesh(v, tr))]))
    out["mesh_torus"] = t
    t = hp.Octree()
    t.FromMemoryBlock(hp.MemoryBlock.frombytes(every_degree_block(hp, out["csg_small"].ToMemoryBlockBytes())))
    out["every_degree"] = t
    # the unit root box, where Query's map is exact
    t = hp.Octree()
    t.Create(hp.Config(target_error_threshold=1e-8, continuity_enforce=0), hp.SdfProgram(CASES["sphere_poly_1e8"]["prog"]))
    out["unit_sphere"] = t
    t = hp.Octree()
    t.FromMemoryBlock(hp.MemoryBlock.frombytes(every_degree_block(hp, out["unit_sphere"].ToMemoryBlockBytes())))
    out["unit_every_degree"] = t
    return out


def user(lv, p):
    """Unit-cube coordinates -> user space (the inverse of Query's map, up to rounding)."""
    return lv.centre + np.asarray(p, np.float64) / lv.inv


def box_sets(lv, seed):
    """Named sets of (lo, hi) boxes in user space: random log-uniform sizes, leaf-face aligned (and 1 ulp off), degenerate,
    straddling the root boundary inside and beyond the L slack, outside, half-spaces, NaN and inverted."""
    rng = np.random.default_rng(seed)
    n = 24
    size = 10.0 ** rng.uniform(-6, 0, (n, 1)) * rng.uniform(0.5, 1.0, (n, 3))
    lo = rng.uniform(-0.5, 0.5, (n, 3)) - size * rng.uniform(0, 1, (n, 3))
    sets = {"random": (user(lv, lo), user(lv, lo + size))}
    pick = rng.choice(len(lv.deg), 8, replace=False)
    size = 2.0 ** -lv.depth[pick, None]
    flo, fhi = user(lv, lv.cell[pick] * size - 0.5), user(lv, (lv.cell[pick] + 1) * size - 0.5)
    sets["leaf_faces"] = (np.concatenate([flo, np.nextafter(flo, -np.inf), np.nextafter(flo, np.inf)]),
                          np.concatenate([fhi, np.nextafter(fhi, np.inf), np.nextafter(fhi, -np.inf)]))
    p = user(lv, rng.uniform(-0.5, 0.5, (6, 3)))
    seg, plane = p.copy(), p.copy()
    seg[:, 0] += 0.1 / lv.inv[0]
    plane[:, :2] += 0.05 / lv.inv[:2]
    sets["degenerate"] = (np.concatenate([p, p, p]), np.concatenate([p, seg, plane]))
    edge = np.array([[0.5 - 1e-3, -0.2, -0.2], [0.5 - 1e-3, -0.2, -0.2], [-0.6, -0.6, -0.6], [0.5 + 2.0 ** -25, 0.1, 0.1], [0.5 + 2.0 ** -24, 0.1, 0.1]])
    ehi = np.array([[0.5 + 2.0 ** -26, -0.1, -0.1], [0.5 + 1e-3, -0.1, -0.1], [0.6, 0.6, 0.6], [0.6, 0.2, 0.2], [0.6, 0.2, 0.2]])
    sets["root_boundary"] = (user(lv, edge), user(lv, ehi))
    sets["outside"] = (user(lv, [[0.7, 0, 0], [-2, -2, -2]]), user(lv, [[0.9, 0.1, 0.1], [-1, 2, 2]]))
    inf = np.inf
    sets["half_spaces"] = (np.array([[-inf, -inf, -inf], [0.0, -inf, -inf], [-inf, -inf, -inf]]), np.array([[inf, inf, inf], [inf, inf, inf], [0.0, inf, inf]]))
    nan = np.nan
    sets["invalid"] = (np.array([[nan, 0, 0], [0.1, 0, 0], [0, 0, 0]]), np.array([[1, 1, 1], [0.0, 1, 1], [1, 1, nan]]))
    return sets


def sample_box(lv, lo, hi, rng, k=400):
    """Corners, face points, random interior points of a box (finite part), and leaf-face points +-1 ulp inside it."""
    lo, hi = np.maximum(lo, user(lv, [-0.6] * 3)), np.minimum(hi, user(lv, [0.6] * 3))
    corners = np.array([[hi[a] if (c >> a) & 1 else lo[a] for a in range(3)] for c in range(8)])
    inner = rng.uniform(lo, hi, (k, 3))
    face = rng.uniform(lo, hi, (k // 2, 3))
    ax = rng.integers(0, 3, len(face))
    face[np.arange(len(face)), ax] = np.where(rng.integers(0, 2, len(face)) == 1, hi[ax], lo[ax])
    cut = inner[: k // 4].copy()
    ax = rng.integers(0, 3, len(cut))
    d = lv.depth.max()
    pu = (cut - lv.centre) * lv.inv
    pu[np.arange(len(cut)), ax] = np.round((pu[np.arange(len(cut)), ax] + 0.5) * 2.0 ** d) / 2.0 ** d - 0.5
    onface = user(lv, pu)
    pts = np.concatenate([corners, inner, face, onface, np.nextafter(onface, np.inf), np.nextafter(onface, -np.inf)])
    return np.clip(pts, lo, hi)


def leaves_of(tree, hp):
    return B.Leaves.from_block(hp.parse_block(tree.ToMemoryBlockBytes()))


@pytest.mark.gpu
@pytest.mark.parametrize("name", TREES)
def test_enclosure_and_checker(hp, trees, name):
    tree = trees[name]
    lv = leaves_of(tree, hp)
    rng = np.random.default_rng(5)
    worst = 0.0
    for kind, (lo, hi) in box_sets(lv, 3).items():
        f_lo, f_hi = tree.QueryBounds(lo, hi)
        for i in range(len(lo)):
            want = lv.bounds(lo[i], hi[i])
            if np.isnan(want[0]) or want[0] == B.DBL_MAX:
                assert np.array_equal([f_lo[i], f_hi[i]], want[:2], equal_nan=True), (kind, i)
                continue
            assert abs(f_lo[i] - want[0]) <= want[2] * (1 + 1e-9), (kind, i, f_lo[i], want)
            assert f_hi[i] == want[1] if want[1] == B.DBL_MAX else abs(f_hi[i] - want[1]) <= want[3] * (1 + 1e-9), (kind, i, f_hi[i], want)
            if want[2] > 0:
                worst = max(worst, abs(f_lo[i] - want[0]) / want[2])
            if not np.isfinite(lo[i]).all() or not np.isfinite(hi[i]).all():
                continue
            pts = sample_box(lv, lo[i], hi[i], rng)
            q = tree.Query(pts)
            assert (q >= f_lo[i]).all() and (q <= f_hi[i]).all(), (kind, i)
            # local minima and maxima of Query from the best samples, through the checker's own polynomial search
            inside = q < B.DBL_MAX
            for sgn in (1.0, -1.0):
                if not inside.any():
                    break
                x0 = pts[inside][np.argmin(sgn * q[inside])]
                blo, bhi = np.maximum(lo[i], user(lv, [-0.5] * 3)), np.minimum(hi[i], user(lv, [0.5] * 3))
                if (blo > bhi).any():
                    break
                r = scipy.optimize.minimize(lambda x: sgn * tree.Query(x[None])[0], x0, method="Powell",
                                            bounds=list(zip(blo, bhi)), options=dict(maxfev=200, xtol=1e-12))
                v = tree.Query(np.clip(r.x, blo, bhi)[None])[0]
                assert f_lo[i] <= v <= f_hi[i], (kind, i)
    print("%s: %d leaves, worst |f_lo - checker| / allowance %.3g" % (name, len(lv.deg), worst))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["unit_sphere", "unit_every_degree"])
def test_structure(hp, trees, name):
    tree = trees[name]
    lv = leaves_of(tree, hp)
    assert (lv.inv == 1.0).all() and (lv.centre == 0.0).all()       # the unit root box: the map is exact
    # [-L, L]^3 and every box containing it: the same f_lo bit for bit; larger boxes have f_hi = DBL_MAX
    big = [B.L, 0.5 + 2.0 ** -24, 0.6, 2.0, np.inf]
    f_lo, f_hi = tree.QueryBounds(-np.array(big)[:, None].repeat(3, 1), np.array(big)[:, None].repeat(3, 1))
    assert len(set(f_lo.view(np.uint64).tolist())) == 1
    assert f_hi[0] < B.DBL_MAX and (f_hi[1:] == B.DBL_MAX).all()
    cells = [lv.interval(i, lv.elo[i], lv.ehi[i]) for i in range(len(lv.deg))]
    lows = np.array([c[0][0] for c in cells])
    j = int(np.argmin(lows))
    assert abs(f_lo[0] - lows[j]) <= cells[j][1] * (1 + 1e-9)
    amax = max(c[1] for c in cells)
    # nesting: octants and nested boxes lie inside the parent box's interval, within the allowance
    rng = np.random.default_rng(9)
    lo = rng.uniform(-0.5, 0.3, (12, 3))
    hi = lo + rng.uniform(0.01, 0.2, (12, 3))
    mid = 0.5 * (lo + hi)
    p_lo, p_hi = tree.QueryBounds(lo, hi)
    for o in range(8):
        sel = np.array([(o >> a) & 1 for a in range(3)], bool)
        c_lo, c_hi = tree.QueryBounds(np.where(sel, mid, lo), np.where(sel, hi, mid))
        assert (c_lo >= p_lo - amax).all() and (c_hi <= p_hi + amax).all()
    n_lo, n_hi = tree.QueryBounds(lo + 0.25 * (hi - lo), hi - 0.3 * (hi - lo))
    assert (n_lo >= p_lo - amax).all() and (n_hi <= p_hi + amax).all()
    # point boxes: strictly inside a leaf, around Query's value, 2 A_leaf wide plus the rounding spread of the leaf's computed
    # Bernstein coefficients (which all equal the value in exact arithmetic and lie within A_leaf of it); on a face, every
    # leaf that meets there
    pick = rng.choice(len(lv.deg), 40, replace=False)
    size = 2.0 ** -lv.depth[pick, None]
    pt = (lv.cell[pick] + rng.uniform(0.1, 0.9, (40, 3))) * size - 0.5
    b_lo, b_hi = tree.QueryBounds(pt, pt)
    q = tree.Query(pt)
    al = np.array([lv.allowance(i) for i in pick])
    assert (b_lo <= q).all() and (q <= b_hi).all() and (b_hi - b_lo <= 4 * al * (1 + 1e-9)).all()
    face = pt.copy()
    face[:, 0] = lv.cell[pick, 0] * size[:, 0] - 0.5
    b_lo, b_hi = tree.QueryBounds(face, face)
    for i in range(len(face)):
        want = lv.bounds(face[i], face[i])
        assert abs(b_lo[i] - want[0]) <= want[2] * (1 + 1e-9) and abs(b_hi[i] - want[1]) <= want[3] * (1 + 1e-9)
        touching = ((lv.ehi >= face[i]) & (lv.elo <= face[i])).all(1).sum()
        assert touching >= 2 or face[i, 0] <= -0.5


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["csg_small", "mesh_torus", "every_degree"])
def test_determinism(hp, trees, name):
    """Host and device entry points, chunked and one-chunk host calls, and a rerun give identical bits."""
    import torch
    tree = trees[name]
    lv = leaves_of(tree, hp)
    rng = np.random.default_rng(21)
    n = 6 * 2 ** 16 + 123
    size = 10.0 ** rng.uniform(-5, -0.5, (n, 1)) * rng.uniform(0.5, 1.0, (n, 3))
    lo = user(lv, rng.uniform(-0.55, 0.55, (n, 3)))
    hi = lo + size / lv.inv
    f_lo, f_hi = tree.QueryBounds(lo, hi)
    g_lo, g_hi = tree.QueryBounds(lo, hi)
    assert np.array_equal(f_lo.view(np.uint64), g_lo.view(np.uint64)) and np.array_equal(f_hi.view(np.uint64), g_hi.view(np.uint64))
    parts = [tree.QueryBounds(lo[s:s + 2 ** 16], hi[s:s + 2 ** 16]) for s in range(0, n, 2 ** 16)]
    assert np.array_equal(np.concatenate([p[0] for p in parts]).view(np.uint64), f_lo.view(np.uint64))
    assert np.array_equal(np.concatenate([p[1] for p in parts]).view(np.uint64), f_hi.view(np.uint64))
    for m in (0, 1, 33, n):
        dl = torch.tensor(lo[:m], dtype=torch.float64, device="cuda")
        dh = torch.tensor(hi[:m], dtype=torch.float64, device="cuda")
        ol = torch.empty(m, dtype=torch.float64, device="cuda")
        oh = torch.empty(m, dtype=torch.float64, device="cuda")
        tree.QueryBoundsDevice(dl.data_ptr(), dh.data_ptr(), m, ol.data_ptr(), oh.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert np.array_equal(ol.cpu().numpy().view(np.uint64), f_lo[:m].view(np.uint64))
        assert np.array_equal(oh.cpu().numpy().view(np.uint64), f_hi[:m].view(np.uint64))
    # a clone builds its own table and gives the same bits
    c_lo, c_hi = tree.copy().QueryBounds(lo[:5000], hi[:5000])
    assert np.array_equal(c_lo.view(np.uint64), f_lo[:5000].view(np.uint64)) and np.array_equal(c_hi.view(np.uint64), f_hi[:5000].view(np.uint64))


@pytest.mark.gpu
def test_argument_errors(hp, trees):
    L = hp.lib()
    t = trees["csg_small"]
    x, v = np.zeros((2, 3)), np.empty(2)
    assert L.hpsdf_query_bounds(None, x.ctypes.data, x.ctypes.data, 2, v.ctypes.data, v.ctypes.data) == hp.ERR_INVALID_ARG
    assert L.hpsdf_query_bounds(t._h, None, x.ctypes.data, 2, v.ctypes.data, v.ctypes.data) == hp.ERR_INVALID_ARG
    assert L.hpsdf_query_bounds(t._h, x.ctypes.data, x.ctypes.data, 2, v.ctypes.data, None) == hp.ERR_INVALID_ARG
    assert L.hpsdf_query_bounds(t._h, None, None, 0, None, None) == hp.OK
    assert L.hpsdf_query_bounds_device(t._h, None, None, 2, None, None, None) == hp.ERR_INVALID_ARG
    assert L.hpsdf_query_bounds_device(t._h, None, None, 0, None, None, None) == hp.OK


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sphere_poly_1e8", "mesh_torus"])
def test_certified_free_blocks(hp, trees, name):
    """Fraction of a 64^3 tiling of the root certified free of the surface; on the sphere no certified block may hold sample
    points of exact distance <= -e and >= +e, e = the largest |Query - exact distance| on a dense sample."""
    tree = trees[name]
    lv = leaves_of(tree, hp)
    k = 64
    e = np.arange(k) / k - 0.5
    g = np.stack(np.meshgrid(e, e, e, indexing="ij"), -1).reshape(-1, 3)
    lo, hi = user(lv, g), user(lv, g + 1.0 / k)
    f_lo, f_hi = tree.QueryBounds(lo, hi)
    free = (f_lo > 0) | (f_hi < 0)
    print("%s: %.4f of the 64^3 blocks certified free of the surface" % (name, free.mean()))
    assert 0.5 < free.mean() < 1.0
    if name != "sphere_poly_1e8":
        return
    c = CASES[name]["prog"]
    assert c[0][0] == "sphere"
    centre, r = np.array(c[0][1][:3]), c[0][1][3]
    exact = lambda x: np.linalg.norm(x - centre, axis=1) - r
    rng = np.random.default_rng(2)
    x = rng.uniform(-0.5, 0.5, (2 ** 20, 3))
    err = np.abs(tree.Query(x) - exact(x)).max()
    sub = (np.stack(np.meshgrid(*[np.linspace(0, 1, 5)] * 3, indexing="ij"), -1).reshape(-1, 3)) / k
    idx = np.nonzero(free)[0]
    pts = (lo[idx][:, None, :] + sub[None]).reshape(-1, 3)
    d = exact(pts).reshape(len(idx), -1)
    assert not ((d <= -err).any(1) & (d >= err).any(1)).any()


@pytest.mark.gpu
def test_cpp_facade(tmp_path):
    exe = str(tmp_path / "bounds_facade_test")
    subprocess.check_call([GXX, "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "bounds_facade_test.cpp"),
                           "-L", os.path.join(PKG, "lib"), "-lhpsdf", "-o", exe])
    env = dict(os.environ, LD_LIBRARY_PATH=os.path.join(PKG, "lib") + ":" + os.environ.get("LD_LIBRARY_PATH", ""))
    out = subprocess.run([exe], env=env, capture_output=True, text=True, timeout=600)
    print(out.stdout)
    assert out.returncode == 0, out.stdout + out.stderr
