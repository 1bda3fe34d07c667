"""hpsdf_query_derivatives / Octree.QueryDerivatives / Octree.QueryTorch: Query's value with the exact gradient and Hessian of
the hit leaf's polynomial (DESIGN §13). Checked against the numpy checker (derivatives_ref.py, itself pinned to the C oracle
on the CPU), against central differences of Query that share nothing with either, against the exact sphere normal, and
through every interface."""
import os
import subprocess

import numpy as np
import pytest

import derivatives_ref as D
from cases import CASES
from common import product_cfg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "hp-adaptive-signed-distance-field-octree_b200")
GXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
EPS = np.finfo(np.float64).eps


# ---- CPU: the checker against the oracle and its own central differences; the entry points without a device ----------------

def every_degree_block(hp, block):
    """`block` with leaf i of degree i % 13 and seeded random coefficients (test_gpu_tree_eval's rewrite)."""
    from test_gpu_tree_eval import rewritten_block
    return rewritten_block(hp, block, collapse=False, seed=13)


def test_checker_values_match_the_oracle(hp, oracle):
    from oracle import hpref
    from cases import root_points
    trees = {}
    for name in ("csg_small", "custom_domain"):
        c = CASES[name]
        trees[name] = (oracle.OracleTree.build(hpref.make_config(threads=8, **c["cfg"]), hpref.make_program(c["prog"]), threads=8), c["cfg"])
    trees["every_degree"] = (oracle.OracleTree.from_block(every_degree_block(hp, trees["csg_small"][0].block().tobytes())),
                             CASES["csg_small"]["cfg"])
    for name, (o, k) in trees.items():
        blk = hp.parse_block(o.block().tobytes())
        pts = root_points(k, 20000, seed=3, margin=0.05)
        val, absum, leaf, _ = D.query_derivatives(blk, pts)
        want = o.query(pts, 8)
        out = leaf < 0
        assert out.any() and (~out).sum() > 14000
        assert np.array_equal(want[out], val["value"][out])
        err = np.abs(val["value"][~out] - want[~out])
        assert (err <= 1e-13 * absum["value"][~out]).all(), (name, (err / absum["value"][~out]).max())
        if name == "every_degree":
            assert set(blk["nodes"]["deg"][leaf[~out]]) == set(range(13))


def test_checker_derivatives_match_its_own_central_differences():
    """Random leaves of every degree: d/du and d2/du2 of the checker against its central differences in leaf coordinates."""
    rng = np.random.default_rng(7)
    h = 1e-5
    for degree in range(13):
        for depth in (0, 4, 10):
            c = rng.normal(size=(1, D.COUNTS[degree])) * 0.5 ** np.arange(D.COUNTS[degree])[None, :] ** 0.5
            u = rng.uniform(-0.99, 0.99, (50, 3))
            cs = np.repeat(c, len(u), 0)
            r, _ = D.eval_leaf(cs, degree, depth, u)
            bi = D.basis_index(degree)
            smax = (np.abs(c[0]) * np.sqrt((2.0 * bi + 1.0) * 2.0 ** depth).prod(1)).sum()     # max |term sum| over the leaf
            for a in range(3):
                e = np.zeros(3); e[a] = h
                rp, _ = D.eval_leaf(cs, degree, depth, u + e)
                rm, _ = D.eval_leaf(cs, degree, depth, u - e)
                # truncation h^2/6 |d3| (Markov bound) + rounding of the differenced values
                bound = lambda k: (h * h / 6 * D.markov(degree, k) + 64 * EPS / h) * smax
                cd = (rp["value"] - rm["value"]) / (2 * h)
                assert np.abs(cd - r["grad"][:, a]).max() <= bound(3), (degree, depth, a)
                for k, (x, y) in enumerate(D.HESS_AXES):
                    if y == a:
                        cdh = (rp["grad"][:, x] - rm["grad"][:, x]) / (2 * h)
                        assert np.abs(cdh - r["hess"][:, k]).max() <= bound(3) * max(D.markov(degree, 1), 1.0) + bound(4), (degree, depth, k)


def test_derivatives_without_a_gpu_fail_with_no_device(hp):
    if hp.device_count() > 0:
        pytest.skip("a GPU is present")
    L = hp.lib()
    x, v, g = np.zeros((2, 3)), np.empty(2), np.empty((2, 3))
    assert L.hpsdf_query_derivatives(None, x.ctypes.data, 2, v.ctypes.data, g.ctypes.data, None) == hp.ERR_NO_DEVICE
    assert L.hpsdf_query_derivatives_device(None, 0, 0, 0, 0, 0, None) == hp.ERR_NO_DEVICE
    for call in (lambda: hp.Octree().QueryDerivatives(np.zeros((2, 3))), lambda: hp.Octree().QueryDerivatives(np.zeros((2, 3)), True),
                 lambda: hp.Octree().QueryDerivativesDevice(0, 0, 0, 0)):
        with pytest.raises(hp.HpsdfError) as e:
            call()
        assert e.value.status == hp.ERR_NO_DEVICE


def test_facade_derivatives_compile_without_a_gpu(tmp_path):
    src = tmp_path / "t.cpp"
    src.write_text('#include "hpsdf.hpp"\nint main() { SDF::Octree t; double x[3] = { 0, 0, 0 }, v = 0, g[3], h[6];\n'
                   'try { t.QueryDerivatives(x, 1, &v, g, h); } catch (const SDF::Error& e) { return e.status == HPSDF_ERR_INVALID_ARG ? 0 : 1; } return 2; }\n')
    exe = str(tmp_path / "t")
    subprocess.check_call([GXX, "-std=c++17", "-I", os.path.join(ROOT, "include"), str(src), "-L", os.path.join(PKG, "lib"), "-lhpsdf", "-o", exe])
    assert subprocess.run([exe], env=dict(os.environ, LD_LIBRARY_PATH=os.path.join(PKG, "lib"))).returncode == 0


def test_package_imports_without_torch():
    """QueryTorch imports torch lazily: importing the package must not."""
    code = ("import sys, importlib; sys.path.insert(0, %r); importlib.import_module('hp-adaptive-signed-distance-field-octree_b200'); "
            "assert 'torch' not in sys.modules" % ROOT)
    subprocess.check_call(["python3", "-c", code])


# ---- GPU: trees and points ----------------------------------------------------------------------------------------------------

TREES = ["csg_small", "c2_csg", "sphere_poly_1e8", "custom_domain", "mesh_torus", "every_degree"]


@pytest.fixture(scope="module")
def trees(hp):
    out = {}
    for name in ("csg_small", "c2_csg", "sphere_poly_1e8", "custom_domain"):
        cfg, prog = product_cfg(hp, name)
        t = hp.Octree()
        t.Create(cfg, prog)
        out[name] = (t, CASES[name]["cfg"])
    from meshgen import bumpy_torus, mesh_root
    v, tr = bumpy_torus(80, 40)
    lo, hi = mesh_root(v)
    t = hp.Octree()
    t.Create(hp.Config(target_error_threshold=1e-6, continuity_enforce=0, root_min=lo, root_max=hi), hp.SdfProgram([("mesh", [], hp.Mesh(v, tr))]))
    out["mesh_torus"] = (t, dict(root_min=tuple(lo), root_max=tuple(hi)))
    t = hp.Octree()
    t.FromMemoryBlock(hp.MemoryBlock.frombytes(every_degree_block(hp, out["csg_small"][0].ToMemoryBlockBytes())))
    out["every_degree"] = (t, CASES["csg_small"]["cfg"])
    return out


def sample_points(hp, tree, k, seed=11):
    """Seeded points in the root extended by 5 % (some outside), points on leaf faces and 1 ulp either side, leaf centres."""
    from cases import root_points
    blk = hp.parse_block(tree.ToMemoryBlockBytes())
    rng = np.random.default_rng(seed)
    uni = root_points(k, 6000, seed, margin=0.05)
    centre, inv = D.root_map(k.get("root_min", (-0.5,) * 3), k.get("root_max", (0.5,) * 3))
    nodes = blk["nodes"]
    leaves = np.nonzero(nodes["deg"] != D.INTERNAL)[0]
    pick = rng.choice(leaves, min(len(leaves), 1500), replace=False)
    mn, mx = nodes["mn"][pick].astype(np.float64), nodes["mx"][pick].astype(np.float64)
    inner = mn + rng.uniform(0.0, 1.0, mn.shape) * (mx - mn)
    face = inner.copy()
    ax = rng.integers(0, 3, len(pick))
    side = rng.integers(0, 2, len(pick))
    face[np.arange(len(pick)), ax] = np.where(side[:, None] == 1, mx, mn)[np.arange(len(pick)), ax]
    face_x = centre + face / inv
    up, down = face_x.copy(), face_x.copy()
    idx = (np.arange(len(pick)), ax)
    up[idx] = np.nextafter(face_x[idx], np.inf)
    down[idx] = np.nextafter(face_x[idx], -np.inf)
    cen = centre + 0.5 * (mn + mx) / inv
    return np.concatenate([uni, face_x, up, down, cen]), blk


def as_tensor(a, torch):
    return torch.tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda")


@pytest.mark.gpu
@pytest.mark.parametrize("name", TREES)
def test_values_bits_and_derivatives_against_the_checker(hp, trees, name):
    import torch
    tree, k = trees[name]
    pts, blk = sample_points(hp, tree, k)
    if name == "every_degree":
        deg = blk["nodes"]["deg"][blk["nodes"]["deg"] != D.INTERNAL]
        print("%s: leaf degrees %s" % (name, np.bincount(deg, minlength=13).tolist()))
        assert (deg <= 6).any() and (deg > 6).any()
    q = tree.Query(pts)
    v1, g1 = tree.QueryDerivatives(pts)
    v2, g2, h2 = tree.QueryDerivatives(pts, hessian=True)
    assert np.array_equal(v1.view(np.uint64), q.view(np.uint64)) and np.array_equal(v2.view(np.uint64), q.view(np.uint64))
    assert np.array_equal(g1.view(np.uint64), g2.view(np.uint64))
    ref, absum, leaf, _ = D.query_derivatives(blk, pts)
    out = leaf < 0
    assert out.any() and (~out).sum() > 5000
    assert (q[out] == D.DBL_MAX).all() and not g2[out].any() and not h2[out].any()
    assert np.signbit(g2[out]).sum() == 0 and np.signbit(h2[out]).sum() == 0
    eg = np.abs(g2 - ref["grad"])[~out]
    eh = np.abs(h2 - ref["hess"])[~out]
    print("%s: %d points, worst |grad - ref| / sum|terms| %.3g, |hess - ref| / sum|terms| %.3g" % (
        name, len(pts), (eg / np.maximum(absum["grad"][~out], 1e-300)).max(), (eh / np.maximum(absum["hess"][~out], 1e-300)).max()))
    assert (eg <= 1e-13 * absum["grad"][~out]).all()
    assert (eh <= 1e-13 * absum["hess"][~out]).all()
    # the device entry point on the current stream: the same bits for n = 0, n not a multiple of 32 and an array that is
    # 8-byte but not 16-byte aligned
    for n in (0, 1, 31, 33, 1000, len(pts)):
        buf = torch.zeros(3 * n + 1, dtype=torch.float64, device="cuda")
        for off in (0, 1):
            x = buf[off:off + 3 * n]
            x.copy_(as_tensor(pts[:n].reshape(-1), torch))
            assert n == 0 or (x.data_ptr() % 16 == 0) == (off == 0)
            dv = torch.empty(n, dtype=torch.float64, device="cuda")
            dg = torch.empty((n, 3), dtype=torch.float64, device="cuda")
            dh = torch.empty((n, 6), dtype=torch.float64, device="cuda")
            s = torch.cuda.current_stream().cuda_stream
            tree.QueryDerivativesDevice(x.data_ptr(), n, dv.data_ptr(), dg.data_ptr(), dh.data_ptr(), stream=s)
            torch.cuda.synchronize()
            assert np.array_equal(dv.cpu().numpy().view(np.uint64), q[:n].view(np.uint64))
            assert np.array_equal(dg.cpu().numpy(), g2[:n]) and np.array_equal(dh.cpu().numpy(), h2[:n])
            tree.QueryDerivativesDevice(x.data_ptr(), n, dv.data_ptr(), dg.data_ptr(), None, stream=s)
            torch.cuda.synchronize()
            assert np.array_equal(dv.cpu().numpy().view(np.uint64), q[:n].view(np.uint64)) and np.array_equal(dg.cpu().numpy(), g2[:n])


def interior_points(hp, tree, k, n, margin, seed):
    """Seeded points inside the root whose local coordinates are at least `margin` of the leaf size from every face."""
    from cases import root_points
    blk = hp.parse_block(tree.ToMemoryBlockBytes())
    pts = root_points(k, 4 * n, seed)
    _, _, leaf, u = D.query_derivatives(blk, pts)
    keep = (leaf >= 0) & (np.abs(u) <= 1.0 - 2.0 * margin).all(1)
    return pts[keep][:n], blk


@pytest.mark.gpu
@pytest.mark.parametrize("name", TREES)
def test_central_differences_of_query(hp, trees, name):
    """Independent of the kernel and the checker: central differences of hpsdf_query in user space with a step of 1e-6 of
    the leaf size (du = 2e-6), at points 1e-3 of the leaf size or more from every face, against grad; the same of grad
    against hess. The bound per component is the sum of
      truncation  du^2 / 6 * Markov(m, 3) * S          (Markov(m, k): V. A. Markov's k-th derivative bound, degree m leaf;
      rounding    (nc + 3m + 3) eps * S / du            S = sum |c_t| NormalisedLength products, max |P| over the leaf)
      position    Markov(m, 1) * S * e_u / du           (e_u: rounding of x +- h and of Query's root map, in u)
    times du/dx; for the Hessian the orders go up by one and the rounding of grad is its checked 1e-13 sum|terms|."""
    tree, k = trees[name]
    pts, blk = interior_points(hp, tree, k, 3000, 1e-3, seed=5)
    assert len(pts) > 1000
    _, g, H = tree.QueryDerivatives(pts, hessian=True)
    leaf, p, inv = D.locate(blk, pts)
    nodes = blk["nodes"]
    deg = nodes["deg"][leaf].astype(np.int64)
    dep = nodes["depth"][leaf].astype(np.int64)
    S = np.zeros(len(pts))
    for i, lf in enumerate(leaf):
        c = blk["coeffs"][int(nodes["cstart"][lf]):int(nodes["cstart"][lf]) + D.COUNTS[deg[i]]]
        bi = D.basis_index(int(deg[i]))
        nl = np.sqrt((2.0 * bi + 1.0) * 2.0 ** dep[i]).prod(1)
        S[i] = (np.abs(c) * nl).sum()
    du = 2e-6
    s = 2.0 ** (dep[:, None] + 1) * inv[None, :]                       # du/dx per axis
    h = du / s
    M = np.array([[D.markov(int(m), kk) for kk in range(5)] for m in deg])
    nc = np.array([D.COUNTS[m] for m in deg])
    e_u = 4 * EPS * (np.abs(p) + np.abs(pts) * inv[None, :] + 1.0) * 2.0 ** (dep[:, None] + 1)
    worst_g = worst_h = 0.0
    for a in range(3):
        e = np.zeros((len(pts), 3)); e[:, a] = h[:, a]
        fp, gp, _ = tree.QueryDerivatives(pts + e, hessian=True)
        fm, gm, _ = tree.QueryDerivatives(pts - e, hessian=True)
        cd = (fp - fm) / (2 * h[:, a])
        bound = (du * du / 6 * M[:, 3] * S + (nc + 3 * deg + 3) * EPS * S / du + M[:, 1] * S * e_u[:, a] / du) * s[:, a]
        err = np.abs(cd - g[:, a])
        worst_g = max(worst_g, (err / bound).max())
        assert (err <= bound).all(), (a, (err / bound).max())
        for kk, (x, y) in enumerate(D.HESS_AXES):
            for (r, c) in ((x, y), (y, x)):
                if c != a:
                    continue
                cdh = (gp[:, r] - gm[:, r]) / (2 * h[:, a])
                m_tr = M[:, 4] if r == c else M[:, 1] * M[:, 3]
                m_pos = M[:, 2] if r == c else M[:, 1] * M[:, 1]
                bnd = (du * du / 6 * m_tr * S + 1e-13 * M[:, 1] * S / du + m_pos * S * e_u[:, a] / du) * s[:, r] * s[:, a]
                errh = np.abs(cdh - H[:, kk])
                worst_h = max(worst_h, (errh / np.maximum(bnd, 1e-300)).max())
                assert (errh <= bnd).all(), (kk, (errh / bnd).max())
    print("%s: central differences within %.3g (grad) and %.3g (hess) of their bounds" % (name, worst_g, worst_h))


@pytest.mark.gpu
def test_sphere_gradient_is_the_exact_normal(hp, trees):
    tree, _ = trees["sphere_poly_1e8"]
    c, r = np.array([0.25, 0.0, 0.0]), 0.5
    rng = np.random.default_rng(19)
    d = rng.normal(size=(100000, 3)); d /= np.linalg.norm(d, axis=1)[:, None]
    x = c + (r + rng.uniform(-0.01, 0.01, (len(d), 1))) * d
    keep = (np.abs(x) < 0.5).all(1)
    x, d = x[keep], d[keep]
    _, g = tree.QueryDerivatives(x)
    mag = np.linalg.norm(g, axis=1)
    ang = np.degrees(np.arccos(np.clip((g * d).sum(1) / mag, -1, 1)))
    print("sphere: %d points within 0.01 of the surface, worst angle to the exact normal %.3g deg, worst | |grad| - 1 | %.3g" %
          (len(x), ang.max(), np.abs(mag - 1).max()))
    assert ang.max() <= 0.5 and np.abs(mag - 1).max() <= 1e-2


# ---- GPU: torch -------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_query_torch(hp, trees):
    import torch
    tree, k = trees["c2_csg"]
    pts, _ = sample_points(hp, tree, k)
    x = as_tensor(pts, torch)
    q = tree.Query(pts)
    assert np.array_equal(tree.QueryTorch(x).cpu().numpy().view(np.uint64), q.view(np.uint64))
    xg = x.clone().requires_grad_(True)
    f = tree.QueryTorch(xg)
    assert np.array_equal(f.detach().cpu().numpy().view(np.uint64), q.view(np.uint64))
    f.sum().backward()
    dv = torch.empty(len(pts), dtype=torch.float64, device="cuda")
    dg = torch.empty((len(pts), 3), dtype=torch.float64, device="cuda")
    tree.QueryDerivativesDevice(x.data_ptr(), len(pts), dv.data_ptr(), dg.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert np.array_equal(xg.grad.cpu().numpy().view(np.uint64), dg.cpu().numpy().view(np.uint64))
    # create_graph: the Hessian-vector product from the ORDER-2 kernel
    xg2 = x[:500].clone().requires_grad_(True)
    (gx,) = torch.autograd.grad(tree.QueryTorch(xg2).sum(), xg2, create_graph=True)
    w = torch.randn_like(gx)
    (hw,) = torch.autograd.grad((gx * w).sum(), xg2)
    _, _, H = tree.QueryDerivatives(pts[:500], hessian=True)
    Hm = H[:, [0, 1, 2, 1, 3, 4, 2, 4, 5]].reshape(-1, 3, 3)
    assert np.allclose(hw.cpu().numpy(), np.einsum("nij,nj->ni", Hm, w.cpu().numpy()), rtol=1e-14, atol=1e-14 * np.abs(Hm).max())
    (gx,) = torch.autograd.grad(tree.QueryTorch(xg2).sum(), xg2, create_graph=True)
    (hx,) = torch.autograd.grad((gx * w).sum(), xg2, create_graph=True)
    with pytest.raises(RuntimeError, match="third derivative"):
        torch.autograd.grad(hx.sum(), xg2)
    # gradcheck / gradgradcheck at points 1e-4 of the leaf size or more inside their leaves (their steps stay in the leaf)
    xi, _ = interior_points(hp, tree, k, 40, 1e-4, seed=23)
    xt = as_tensor(xi, torch).requires_grad_(True)
    assert torch.autograd.gradcheck(tree.QueryTorch, (xt,), eps=1e-7, atol=1e-6, rtol=1e-6)
    assert torch.autograd.gradgradcheck(tree.QueryTorch, (xt,), eps=1e-7, atol=1e-5, rtol=1e-5)
    # nothing is copied silently
    for bad in (x.float(), x.cpu(), x[:, :2].contiguous(), x.reshape(-1), x.t().contiguous().t()):
        with pytest.raises((TypeError, ValueError)):
            tree.QueryTorch(bad)
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            tree.QueryTorch(x.to("cuda:1"))


@pytest.mark.gpu
def test_argument_errors(hp, trees):
    import torch
    tree, _ = trees["csg_small"]
    L = hp.lib()
    x, v, g, hh = np.zeros((4, 3)), np.empty(4), np.empty((4, 3)), np.empty((4, 6))
    call = lambda t=tree._h, xx=x.ctypes.data, vv=v.ctypes.data, gg=g.ctypes.data, hs=hh.ctypes.data, n=4: L.hpsdf_query_derivatives(t, xx, n, vv, gg, hs)
    assert call() == hp.OK and call(hs=None) == hp.OK and call(n=0, xx=None, vv=None, gg=None) == hp.OK
    for bad in (dict(t=None), dict(xx=None), dict(vv=None), dict(gg=None)):
        assert call(**bad) == hp.ERR_INVALID_ARG, bad
    dx = torch.zeros((4, 3), dtype=torch.float64, device="cuda")
    dv = torch.empty(4, dtype=torch.float64, device="cuda")
    dg = torch.empty((4, 3), dtype=torch.float64, device="cuda")
    assert L.hpsdf_query_derivatives_device(tree._h, dx.data_ptr(), 4, dv.data_ptr(), dg.data_ptr(), None, None) == hp.OK
    assert L.hpsdf_query_derivatives_device(tree._h, None, 4, dv.data_ptr(), dg.data_ptr(), None, None) == hp.ERR_INVALID_ARG
    assert L.hpsdf_query_derivatives_device(tree._h, dx.data_ptr(), 4, dv.data_ptr(), None, None, None) == hp.ERR_INVALID_ARG
    assert L.hpsdf_query_derivatives_device(None, dx.data_ptr(), 4, dv.data_ptr(), dg.data_ptr(), None, None) == hp.ERR_INVALID_ARG
    torch.cuda.synchronize()
    if hp.device_count() > 1:
        other = 1 if torch.cuda.current_device() == 0 else 0
        with torch.cuda.device(other):
            assert L.hpsdf_query_derivatives_device(tree._h, dx.data_ptr(), 4, dv.data_ptr(), dg.data_ptr(), None, None) == hp.ERR_INVALID_ARG


FACADE_SRC = r"""
#include <cstdio>
#include "hpsdf.hpp"
int main()
{
    SDF::Config cfg;
    cfg.targetErrorThreshold = 1e-8;
    cfg.continuity.enforce = false;
    SDF::Octree tree;
    tree.Create(cfg, SDF::Program().Sphere(0.05, -0.02, 0.01, 0.3));
    const double x[3] = { 0.3, 0.1, -0.2 };
    double v, g[3], h[6];
    tree.QueryDerivatives(x, 1, &v, g, h);
    std::printf("%.17g %.17g %.17g %.17g %.17g %.17g %.17g %.17g %.17g %.17g\n", v, g[0], g[1], g[2], h[0], h[1], h[2], h[3], h[4], h[5]);
    return 0;
}
"""


@pytest.mark.gpu
def test_cpp_facade(tmp_path):
    src, exe = tmp_path / "d.cpp", str(tmp_path / "d")
    src.write_text(FACADE_SRC)
    subprocess.check_call([GXX, "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), str(src), "-L", os.path.join(PKG, "lib"), "-lhpsdf", "-o", exe])
    env = dict(os.environ, LD_LIBRARY_PATH=os.path.join(PKG, "lib") + ":" + os.environ.get("LD_LIBRARY_PATH", ""))
    out = subprocess.run([exe], env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    v, *rest = [float(t) for t in out.stdout.split()]
    g, h = np.array(rest[:3]), np.array(rest[3:])
    y = np.array([0.3, 0.1, -0.2]) - np.array([0.05, -0.02, 0.01])
    r = np.linalg.norm(y)
    assert abs(v - (r - 0.3)) <= 1e-6 and np.abs(g - y / r).max() <= 1e-4
    Hm = (np.eye(3) - np.outer(y, y) / r ** 2) / r         # the exact sphere's; the 1e-8 tree's differs by about 1e-2
    assert np.abs(h - Hm[[0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2]]).max() <= 5e-2
