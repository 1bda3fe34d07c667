"""hpsdf_raycast / Octree.Raycast: first crossings of F = iso along rays, exact per leaf (DESIGN §12). Checked against the
analytic answer on plane trees (degenerate rays included), against the independent numpy checker (raycast_ref.py) on
analytic and mesh-sourced trees, against the exact sphere, and through every interface."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import raycast_ref as R
from cases import CASES
from common import product_cfg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "hp-adaptive-signed-distance-field-octree_b200")
GXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"


# ---- CPU: the checker itself on exactly polynomial fields, and the entry points without a device ----------------------------

def box_grid(k=4):
    e = np.arange(k) / k - 0.5
    lo = np.stack(np.meshgrid(e, e, e, indexing="ij"), -1).reshape(-1, 3)
    return lo, lo + 1.0 / k


def analytic_first_root(o, d, f_quad, iso):
    """First t >= ta in the unit cube with f(o + t d) <= iso, f = (A, b, c): p.A.p + b.p + c."""
    A, b, c = f_quad
    c2 = d @ A @ d
    c1 = 2 * o @ A @ d + b @ d
    c0 = o @ A @ o + b @ o + c - iso
    cl = R.clip(o, d, 0.0, np.inf)
    if cl is None:
        return np.inf
    ta, tb = cl
    if c2 * ta * ta + c1 * ta + c0 <= 0:
        return ta
    roots = np.roots([c2, c1, c0]) if abs(c2) > 0 else (np.array([-c0 / c1]) if c1 else np.array([]))
    roots = sorted(r.real for r in np.atleast_1d(roots) if abs(r.imag) < 1e-12 and ta <= r.real <= tb)
    return roots[0] if roots else np.inf


@pytest.mark.parametrize("kind", ["sphere", "plane"])
def test_checker_reproduces_analytic_first_roots(kind):
    rng = np.random.default_rng(3)
    if kind == "sphere":
        f = (np.eye(3), np.zeros(3), -0.3 ** 2)
    else:
        nrm = np.array([0.3, -0.5, 0.81]) / np.linalg.norm([0.3, -0.5, 0.81])
        f = (np.zeros((3, 3)), nrm, -0.05)
    lo, hi = box_grid(4)
    deg = np.full(len(lo), 2 if kind == "sphere" else 1)
    ev = lambda P: np.einsum("ni,ij,nj->n", P, f[0], P) + P @ f[1] + f[2]
    o = np.concatenate([rng.uniform(-0.5, 0.5, (150, 3)), rng.uniform(-1.5, 1.5, (150, 3))])
    d = rng.normal(size=(300, 3)) * rng.uniform(0.2, 3.0, (300, 1))
    for iso in (0.0, 0.02):
        got = R.cast(o, d, (-0.5,) * 3, (0.5,) * 3, lo, hi, deg, ev, iso=iso, scale=np.sqrt(3))
        want = np.array([analytic_first_root(o[i], d[i], f, iso) for i in range(len(o))])
        assert np.array_equal(np.isfinite(got["t"]), np.isfinite(want))
        fin = np.isfinite(want)
        assert fin.sum() > 30
        assert np.abs(got["t"][fin] - want[fin]).max() <= 1e-12


def test_raycast_without_a_gpu_fails_with_no_device(hp):
    if hp.device_count() > 0:
        pytest.skip("a GPU is present")
    for call in (lambda: hp.Octree().Raycast(np.zeros((2, 3)), np.ones((2, 3))),
                 lambda: hp.Octree().RaycastDevice(0, 0, 0, 0)):
        with pytest.raises(hp.HpsdfError) as e:
            call()
        assert e.value.status == hp.ERR_NO_DEVICE


def test_facade_raycast_compiles_without_a_gpu(tmp_path):
    src = tmp_path / "t.cpp"
    src.write_text('#include "hpsdf.hpp"\nint main() { SDF::Octree t; double o[3] = { 0, 0, 0 }, d[3] = { 1, 0, 0 }, th = 0, n[3];\n'
                   'try { t.Raycast(o, d, 1, 0.0, 1e30, 0.0, &th, n); } catch (const SDF::Error& e) { return e.status == HPSDF_ERR_INVALID_ARG ? 0 : 1; } return 2; }\n')
    exe = str(tmp_path / "t")
    subprocess.check_call([GXX, "-std=c++17", "-I", os.path.join(ROOT, "include"), str(src), "-L", os.path.join(PKG, "lib"), "-lhpsdf", "-o", exe])
    assert subprocess.run([exe], env=dict(os.environ, LD_LIBRARY_PATH=os.path.join(PKG, "lib"))).returncode == 0


# ---- GPU: plane trees against the analytic answer ----------------------------------------------------------------------------

PLANE_N = np.array([0.3, -0.5, 0.81]) / np.linalg.norm([0.3, -0.5, 0.81])
PLANE_D = 0.07
ROOTS = {"default": ((-0.5,) * 3, (0.5,) * 3), "custom": ((-0.3, -0.7, -0.2), (1.1, 0.6, 0.9))}


@pytest.fixture(scope="module")
def plane_trees(hp):
    out = {}
    for name, (lo, hi) in ROOTS.items():
        t = hp.Octree()
        t.Create(hp.Config(target_error_threshold=1e-8, continuity_enforce=0, root_min=lo, root_max=hi),
                 hp.SdfProgram([("plane", list(PLANE_N) + [PLANE_D])]))
        out[name] = t
    return out


def plane_expected(o, d, root, iso, t_min=0.0, t_max=np.inf):
    """The tree's field is the plane composed with Create's sampling map x = centre + p sizes (f32 widened), while Query maps
    p = (x - centre) invSizes: linear in p, so the crossing along p0 + t dp is solved exactly in closed form."""
    centre, inv = R.root_map(*root)
    mn, mx = np.asarray(root[0], np.float32), np.asarray(root[1], np.float32)
    sizes = (mx - mn).astype(np.float64)
    out = np.full(len(o), np.inf)
    for i in range(len(o)):
        if not (np.isfinite(o[i]).all() and np.isfinite(d[i]).all()) or not d[i].any():
            continue
        p0, dp = (o[i] - centre) * inv, d[i] * inv
        cl = R.clip(p0, dp, t_min, t_max)
        if cl is None:
            continue
        ta, tb = cl
        f = lambda t: PLANE_N @ (centre + (p0 + t * dp) * sizes) - PLANE_D - iso
        if f(ta) <= 0:
            out[i] = ta
            continue
        slope = PLANE_N @ (dp * sizes)
        if slope < 0:
            tc = ta - f(ta) / slope
            if tc <= tb:
                out[i] = tc
    return out


def plane_rays(root, rng, n=3000):
    lo, hi = (np.asarray(x, np.float64) for x in root)
    size = hi - lo
    o = np.concatenate([rng.uniform(lo, hi, (n // 2, 3)), rng.uniform(lo - 0.6 * size, hi + 0.6 * size, (n - n // 2, 3))])
    d = rng.uniform(lo, hi, (n, 3)) - o
    d *= rng.uniform(0.3, 3.0, (n, 1))
    # parallel to the plane: inside (t = ta) or outside (a miss)
    par = np.cross(PLANE_N, rng.normal(size=(200, 3)))
    po = rng.uniform(lo, hi, (200, 3))
    return np.concatenate([o, po]), np.concatenate([d, par])


def assert_plane(got, want, root):
    diag = np.linalg.norm(np.asarray(root[1]) - np.asarray(root[0]))
    assert np.array_equal(np.isfinite(got), np.isfinite(want)), np.nonzero(np.isfinite(got) != np.isfinite(want))[0][:10]
    return diag


@pytest.mark.gpu
@pytest.mark.parametrize("root", ["default", "custom"])
@pytest.mark.parametrize("iso", [0.0, 0.03, -0.02])
def test_plane_tree_is_exact(plane_trees, root, iso):
    rng = np.random.default_rng(17)
    o, d = plane_rays(ROOTS[root], rng)
    t, nrm = plane_trees[root].Raycast(o, d, iso=iso)
    want = plane_expected(o, d, ROOTS[root], iso)
    diag = assert_plane(t, want, ROOTS[root])
    fin = np.isfinite(want)
    assert fin.sum() > 1000 and (~fin).sum() > 50
    err = np.abs(t[fin] - want[fin]) * np.linalg.norm(d[fin], axis=1)
    assert err.max() <= 1e-12 * diag, err.max() / diag
    # normals: the plane's gradient mapped to user space, unit length
    centre, inv = R.root_map(*ROOTS[root])
    sizes = (np.asarray(ROOTS[root][1], np.float32) - np.asarray(ROOTS[root][0], np.float32)).astype(np.float64)
    g = PLANE_N * sizes * inv
    g /= np.linalg.norm(g)
    assert np.abs(nrm[fin] - g).max() <= 1e-9
    assert not nrm[~fin].any()


@pytest.mark.gpu
@pytest.mark.parametrize("iso", [0.0, 0.03])
def test_plane_tree_degenerate_rays(plane_trees, iso):
    root = ROOTS["default"]
    o, d = [], []
    for ax in range(3):                                    # axis-aligned, both senses, from inside and outside
        for s in (1.0, -1.0):
            e = np.zeros(3); e[ax] = s
            for start in ((0.1, -0.2, 0.3), (-0.8, 0.0, 0.0), (0.0, 0.9, -0.1), (0.3, 0.3, -0.7)):
                o.append(start); d.append(e)
    for y in (0.125, 0.25, -0.0625, 0.0):                  # inside cell face planes (dyadic coordinates, no motion along them)
        for z in (0.25, -0.375, 0.0):
            o.append((-0.7, y, z)); d.append((1.0, 0.0, 0.0))
            o.append((0.6, y, z)); d.append((-1.0, 0.0, 0.0))
            o.append((y, -0.8, z)); d.append((0.0, 1.0, 0.0))
    for start in ((-0.625, -0.625, -0.625), (0.0625, -0.125, 0.1875), (-0.5, -0.5, -0.5), (0.5, 0.5, 0.5)):   # edges, corners
        for dd in ((1, 1, 1), (-1, -1, -1), (1, 1, 0), (0, -1, 1), (1, -1, 1)):
            o.append(start); d.append(dd)
    o.append((0.1, 0.1, 0.1)); d.append((0.0, 0.0, 0.0))
    o.append((0.1, 0.1, 0.1)); d.append((np.nan, 1.0, 0.0))
    o.append((np.inf, 0.1, 0.1)); d.append((1.0, 0.0, 0.0))
    o, d = np.asarray(o, np.float64), np.asarray(d, np.float64)
    tree = plane_trees["default"]
    t, _ = tree.Raycast(o, d, iso=iso)
    want = plane_expected(o, d, root, iso)
    assert_plane(t, want, root)
    fin = np.isfinite(want)
    assert fin.sum() > 30
    assert np.abs(t[fin] - want[fin]).max() * np.abs(d[fin]).max() <= 1e-12 * np.sqrt(3)
    assert not np.isfinite(t[-3:]).any()
    # t_min beyond the first crossing and t_max before it
    hit = np.nonzero(fin & (want > 0.05))[0]
    tmin = float(want[hit].max()) + 1e-3
    t2, _ = tree.Raycast(o[hit], d[hit], t_min=tmin, iso=iso)
    w2 = plane_expected(o[hit], d[hit], root, iso, t_min=tmin)
    assert_plane(t2, w2, root)
    f2 = np.isfinite(w2)
    assert np.abs(t2[f2] - w2[f2]).max() <= 1e-9
    t3, _ = tree.Raycast(o[hit], d[hit], t_max=float(want[hit].min()) * 0.5, iso=iso)
    w3 = plane_expected(o[hit], d[hit], root, iso, t_max=float(want[hit].min()) * 0.5)
    assert_plane(t3, w3, root)


# ---- GPU: analytic and mesh-sourced trees against the checker ------------------------------------------------------------------

@pytest.fixture(scope="module")
def trees(hp):
    out = {}
    for name in ("sphere_poly_1e8", "custom_domain", "c2_csg", "csg_small"):
        cfg, prog = product_cfg(hp, name)
        t = hp.Octree()
        t.Create(cfg, prog)
        out[name] = t
    return out


def root_of(name):
    k = CASES[name]["cfg"]
    return k.get("root_min", (-0.5,) * 3), k.get("root_max", (0.5,) * 3)


def seeded_rays(root, n, seed):
    """Half from inside the root, half from a shell around it, aimed at random points of the root."""
    rng = np.random.default_rng(seed)
    lo, hi = (np.asarray(x, np.float64) for x in root)
    size = hi - lo
    inside = rng.uniform(lo, hi, (n // 2, 3))
    outside = rng.uniform(lo - 0.5 * size, hi + 0.5 * size, (4 * n, 3))
    outside = outside[((outside < lo) | (outside > hi)).any(1)][: n - n // 2]
    o = np.concatenate([inside, outside])
    d = (rng.uniform(lo, hi, (n, 3)) - o) * rng.uniform(0.5, 2.0, (n, 1))
    return o, d


def compare_with_checker(hp, tree, root, o, d, iso, label):
    t, nrm = tree.Raycast(o, d, iso=iso)
    lo, hi, deg = R.tree_leaves(hp.parse_block(tree.ToMemoryBlockBytes()))
    diag = float(np.linalg.norm(np.asarray(root[1], np.float64) - np.asarray(root[0], np.float64)))
    ref = R.cast(o, d, root[0], root[1], lo, hi, deg, tree.Query, iso=iso, scale=diag)
    ok = ref["flag"] == 0
    excluded = 1.0 - ok.mean()
    print("%s iso %g: %d rays, %d hits, excluded %.2f %% (near-tangent / near-touch %d, ambiguous fit %d)" %
          (label, iso, len(o), np.isfinite(ref["t"]).sum(), 100 * excluded, (ref["flag"] == 1).sum(), (ref["flag"] == 2).sum()))
    assert excluded <= 0.02
    bad = np.isfinite(t[ok]) != np.isfinite(ref["t"][ok])
    assert not bad.any(), np.nonzero(ok)[0][bad][:10]
    hit = ok & np.isfinite(ref["t"])
    err = np.abs(t[hit] - ref["t"][hit]) * np.linalg.norm(d[hit], axis=1)
    assert err.max() <= 1e-9 * diag, err.max() / diag
    assert not nrm[~np.isfinite(t)].any()
    return t, nrm, ref, ok, diag


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sphere_poly_1e8", "custom_domain", "c2_csg", "csg_small"])
@pytest.mark.parametrize("iso_frac", [0.0, 0.015])
def test_analytic_trees_against_the_checker(hp, trees, name, iso_frac):
    root = root_of(name)
    o, d = seeded_rays(root, 2000, seed=29)
    iso = iso_frac * (root[1][0] - root[0][0])
    t, _, ref, ok, _ = compare_with_checker(hp, trees[name], root, o, d, iso, name)
    assert np.isfinite(t).sum() > 200


@pytest.mark.gpu
def test_sphere_against_the_exact_intersection(hp, trees):
    tree = trees["sphere_poly_1e8"]
    c, r = np.array([0.25, 0.0, 0.0]), 0.5
    rng = np.random.default_rng(41)
    # the tree's surface error, measured on the exact sphere (inside the root)
    u = rng.normal(size=(200000, 3)); u /= np.linalg.norm(u, axis=1)[:, None]
    s = c + r * u
    s = s[(np.abs(s) <= 0.5).all(1)]
    e_s = np.abs(tree.Query(s)).max()
    o = rng.uniform(-0.5, 0.5, (20000, 3))
    o = o[np.linalg.norm(o - c, axis=1) > r][:4000]
    tgt = c + r * rng.uniform(-0.6, 0.6, (len(o), 3))
    d = tgt - o
    t, nrm = tree.Raycast(o, d)
    # exact first intersection with the sphere (|o + t d - c| = r), kept when it lies inside the root and is transversal
    oc = o - c
    a, b, cc = (d * d).sum(1), 2 * (oc * d).sum(1), (oc * oc).sum(1) - r * r
    disc = b * b - 4 * a * cc
    te = np.where(disc > 0, (-b - np.sqrt(np.maximum(disc, 0))) / (2 * a), np.inf)
    x = o + te[:, None] * d
    n_ex = (x - c) / r
    cos = np.abs((n_ex * d).sum(1)) / np.linalg.norm(d, axis=1)
    use = (disc > 0) & (te > 0) & (np.abs(x) <= 0.5).all(1) & (cos >= 0.3)
    assert use.sum() > 1000
    assert np.isfinite(t[use]).all()
    bound = 2.0 * e_s / cos[use]                          # a surface error e_s moves a crossing by e_s / cos along the ray
    err = np.abs(t[use] - te[use]) * np.linalg.norm(d[use], axis=1)
    print("sphere: surface error %.3g, worst |dt||d| %.3g of its bound" % (e_s, (err / bound).max()))
    assert (err <= bound).all()
    ang = np.degrees(np.arccos(np.clip((nrm[use] * n_ex[use]).sum(1), -1, 1)))
    print("sphere: normals within %.3g deg of the exact normal" % ang.max())
    assert ang.max() <= 1.0
    # against central differences of Query inside the hit leaf. Every leaf face lies on the 2^-10 grid of the unit cube (the
    # default root maps user space to it unchanged), so points farther than 4h from that grid on every axis keep x +- h e_k
    # in their leaf. (QueryWithGradient is no yardstick here: it mirrors the reference's FApproxWithGradient, which
    # differences only the Legendre factor of axis k and drops the other two factors of every basis function.)
    h = 1e-7
    xh = o[use] + t[use][:, None] * d[use]
    off = (xh + 0.5) * 1024.0
    inner = (np.abs(off - np.round(off)) / 1024.0 > 4 * h).all(1)
    assert inner.mean() >= 0.9
    xh, nh = xh[inner], nrm[use][inner]
    g = np.stack([(tree.Query(xh + h * e) - tree.Query(xh - h * e)) / (2 * h) for e in np.eye(3)], 1)
    g /= np.linalg.norm(g, axis=1)[:, None]
    ang_cd = np.degrees(np.arccos(np.clip((nh * g).sum(1), -1, 1)))
    print("sphere: normals within %.3g deg of central differences of Query (h = %g) on %d hits" % (ang_cd.max(), h, len(xh)))
    assert ang_cd.max() <= 1e-3


@pytest.mark.gpu
def test_mesh_tree_pinhole_camera(hp):
    from meshgen import bumpy_torus, mesh_root
    verts, tris = bumpy_torus(200, 90)
    lo, hi = mesh_root(verts)
    tree = hp.Octree()
    tree.Create(hp.Config(target_error_threshold=1e-6, continuity_enforce=0, root_min=lo, root_max=hi), hp.SdfProgram([("mesh", [], hp.Mesh(verts, tris))]))
    lo, hi = np.asarray(lo), np.asarray(hi)
    centre, ext = (lo + hi) / 2, (hi - lo).max()
    o, d = pinhole(centre + ext * np.array([0.35, -0.9, 0.55]), centre, 256, 0.45)
    t, nrm = tree.Raycast(o, d)
    print("pinhole 256^2: hit fraction %.3f" % np.isfinite(t).mean())
    assert 0.1 < np.isfinite(t).mean() < 0.95
    pick = np.random.default_rng(2).choice(len(o), 2000, replace=False)
    ts, _, ref, ok, diag = compare_with_checker(hp, tree, (tuple(lo), tuple(hi)), o[pick], d[pick], 0.0, "bumpy torus")
    assert np.array_equal(ts, t[pick])
    trans = ok & np.isfinite(ref["t"]) & ~ref["at_entry"]
    q = tree.Query(o[pick][trans] + t[pick][trans][:, None] * d[pick][trans])
    assert np.abs(q).max() <= 1e-9 * diag


def pinhole(eye, target, res, fov):
    """Primary rays of a res x res pinhole camera at `eye` looking at `target`, half-angle `fov` (radians)."""
    f = target - eye; f /= np.linalg.norm(f)
    r = np.cross(f, [0.0, 0.0, 1.0]); r /= np.linalg.norm(r)
    u = np.cross(r, f)
    s = np.tan(fov) * ((np.arange(res) + 0.5) / res * 2 - 1)
    X, Y = np.meshgrid(s, s)
    d = f[None, :] + X.reshape(-1, 1) * r[None, :] + Y.reshape(-1, 1) * u[None, :]
    return np.broadcast_to(eye, d.shape).copy(), d


# ---- GPU: interfaces ----------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_device_form_block_copy_and_scaling(hp, trees):
    import torch
    tree = trees["c2_csg"]
    root = root_of("c2_csg")
    o, d = seeded_rays(root, 5000, seed=5)
    t, nrm = tree.Raycast(o, d, iso=0.004)
    assert np.isfinite(t).sum() > 500
    t2, n2 = tree.Raycast(o, d, iso=0.004)
    assert np.array_equal(t, t2) and np.array_equal(nrm, n2)
    do, dd = torch.tensor(o, device="cuda"), torch.tensor(d, device="cuda")
    dt, dn = torch.empty(len(o), dtype=torch.float64, device="cuda"), torch.empty((len(o), 3), dtype=torch.float64, device="cuda")
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        tree.RaycastDevice(do.data_ptr(), dd.data_ptr(), len(o), dt.data_ptr(), dn.data_ptr(), iso=0.004, stream=side.cuda_stream)
    side.synchronize()
    assert np.array_equal(dt.cpu().numpy(), t) and np.array_equal(dn.cpu().numpy(), nrm)
    tree.RaycastDevice(do.data_ptr(), dd.data_ptr(), len(o), dt.data_ptr(), None, iso=0.004)      # normals optional
    torch.cuda.synchronize()
    assert np.array_equal(dt.cpu().numpy(), t)
    copy = hp.Octree()
    mb = tree.ToMemoryBlock()
    try:
        copy.FromMemoryBlock(mb)
    finally:
        mb.free()
    t3, n3 = copy.Raycast(o, d, iso=0.004)
    assert np.array_equal(t3, t) and np.array_equal(n3, nrm)
    for k in (3.0, 0.125, 7.3):
        tk, _ = tree.Raycast(o, d * k, iso=0.004)
        fin = np.isfinite(t)
        assert np.array_equal(np.isfinite(tk), fin)
        assert np.abs(tk[fin] * k - t[fin]).max() <= 1e-12 * np.abs(t[fin]).max()


@pytest.mark.gpu
def test_argument_errors(hp, trees):
    import torch
    tree = trees["c2_csg"]
    L = hp.lib()
    o = np.zeros((4, 3)); d = np.ones((4, 3)); t = np.empty(4); n = np.empty((4, 3))
    def call(tmin=0.0, tmax=np.inf, iso=0.0, oo=o.ctypes.data, dd=d.ctypes.data, tt=t.ctypes.data, nn=n.ctypes.data, h=tree._h, cnt=4):
        return L.hpsdf_raycast(h, oo, dd, cnt, tmin, tmax, iso, tt, nn)
    assert call() == hp.OK and call(nn=None) == hp.OK and call(tmax=5.0) == hp.OK
    assert call(cnt=0, oo=None, dd=None, tt=None) == hp.OK
    for bad in (dict(oo=None), dict(dd=None), dict(tt=None), dict(h=None), dict(tmin=np.nan), dict(tmin=-np.inf), dict(tmin=np.inf),
                dict(iso=np.nan), dict(iso=np.inf), dict(tmax=np.nan), dict(tmin=1.0, tmax=0.5)):
        assert call(**bad) == hp.ERR_INVALID_ARG, bad
    do = torch.zeros((4, 3), dtype=torch.float64, device="cuda")
    dt = torch.empty(4, dtype=torch.float64, device="cuda")
    assert L.hpsdf_raycast_device(tree._h, do.data_ptr(), do.data_ptr(), 4, 0.0, np.inf, 0.0, dt.data_ptr(), None, None) == hp.OK
    assert L.hpsdf_raycast_device(tree._h, do.data_ptr(), do.data_ptr(), 4, 0.0, -1.0, 0.0, dt.data_ptr(), None, None) == hp.ERR_INVALID_ARG
    assert L.hpsdf_raycast_device(tree._h, None, do.data_ptr(), 4, 0.0, 1.0, 0.0, dt.data_ptr(), None, None) == hp.ERR_INVALID_ARG
    torch.cuda.synchronize()
    if hp.device_count() < 2:
        return
    other = 1 if torch.cuda.current_device() == 0 else 0
    with torch.cuda.device(other):
        assert L.hpsdf_raycast_device(tree._h, do.data_ptr(), do.data_ptr(), 4, 0.0, 1.0, 0.0, dt.data_ptr(), None, None) == hp.ERR_INVALID_ARG


FACADE_SRC = r"""
#include <cstdio>
#include "hpsdf.hpp"
int main(int argc, char** argv)
{
    SDF::Config cfg;
    cfg.targetErrorThreshold = 1e-7;
    cfg.continuity.enforce = false;
    SDF::Octree tree;
    tree.Create(cfg, SDF::Program().Sphere(0.05, -0.02, 0.01, 0.3));
    const double o[6] = { -0.9, 0.0, 0.0, 0.4, 0.45, -0.45 }, d[6] = { 1.0, 0.0, 0.0, -1.0, -1.0, 1.0 };
    double t[2], n[6];
    tree.Raycast(o, d, 2, 0.0, 1e300, 0.0, t, n);
    std::printf("%.17g %.17g %.17g %.17g %.17g\n", t[0], t[1], n[0], n[1], n[2]);
    return 0;
}
"""


@pytest.mark.gpu
def test_cpp_facade_matches_the_python_call(hp, tmp_path):
    src, exe = tmp_path / "ray.cpp", str(tmp_path / "ray")
    src.write_text(FACADE_SRC)
    subprocess.check_call([GXX, "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), str(src), "-L", os.path.join(PKG, "lib"), "-lhpsdf", "-o", exe])
    env = dict(os.environ, LD_LIBRARY_PATH=os.path.join(PKG, "lib") + ":" + os.environ.get("LD_LIBRARY_PATH", ""))
    out = subprocess.run([exe], env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    t0, t1, nx, ny, nz = [float(x) for x in out.stdout.split()]
    assert abs(t0 - (0.9 + 0.05 - np.sqrt(0.3 ** 2 - 0.02 ** 2 - 0.01 ** 2))) <= 1e-4
    assert abs(np.linalg.norm([nx, ny, nz]) - 1.0) <= 1e-12 and nx < -0.99
    # the second ray, (0.4, 0.45, -0.45) + t (-1, -1, 1), passes 0.094 from the centre: its first crossing solves
    # 3 t^2 - 2 b t + c = 0 with b = 0.35 + 0.47 + 0.46 and c = 0.35^2 + 0.47^2 + 0.46^2 - 0.3^2
    b, c = 0.35 + 0.47 + 0.46, 0.35 ** 2 + 0.47 ** 2 + 0.46 ** 2 - 0.3 ** 2
    assert abs(t1 - (b - np.sqrt(b * b - 3 * c)) / 3) <= 1e-4
