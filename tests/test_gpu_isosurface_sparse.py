"""hpsdf_extract_isosurface_sparse / Octree.ExtractIsosurfaceSparse: the mesh of hpsdf_extract_isosurface, bit for bit and in
the same order, on grids of up to 16384 cells per axis (DESIGN §15). Both entry points take the dense pipeline below a
grid-point crossover and the sparse one above it, and always the sparse one when an axis has more than 1024 cells; the
sparse pipeline's cases are therefore grids with such an axis. Checked against the numpy checker (isosurface_ref.py), the
plane-by-plane torch checker (isosurface_slab_ref.py), and as a mesh at 4096³."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import isosurface_ref as R
import isosurface_slab_ref as S
from cases import CASES
from common import product_cfg
from test_gpu_isosurface import GXX, PKG, ROOT, root_box, sphere_field


def assert_identical(got, want):
    (gv, gt), (wv, wt) = got, want
    assert gv.dtype == np.float32 and gt.dtype == np.uint32
    assert gv.shape == wv.shape and gt.shape == wt.shape
    assert np.array_equal(gv.view(np.uint32), wv.view(np.uint32))
    assert np.array_equal(gt, wt)


# ---- CPU: the slab checker against the numpy checker, and the entry point without a device -----------------------------

def torus_field(P):
    return np.sqrt((np.sqrt(P[:, 0] ** 2 + P[:, 1] ** 2) - 0.3) ** 2 + P[:, 2] ** 2) - 0.1


@pytest.mark.parametrize("field, n, lo, hi, iso", [
    (sphere_field, (20, 24, 28), (-0.5,) * 3, (0.5,) * 3, 0.0),
    (sphere_field, (37, 16, 17), (-0.4, -0.5, -0.45), (0.45, 0.5, 0.3), 0.02),
    (torus_field, (33, 17, 41), (-0.45, -0.5, -0.3), (0.5, 0.41, 0.3), 0.01),
    (torus_field, (48, 40, 2), (-0.5,) * 3, (0.5, 0.5, 0.02), 0.0),
    (sphere_field, (1, 1, 1), (-0.5,) * 3, (0.5,) * 3, 0.3),
])
def test_slab_checker_equals_the_numpy_checker(field, n, lo, hi, iso):
    want = R.extract(field(R.grid_points(n, lo, hi)), n, lo, hi, iso)
    v, t = S.extract(S.numpy_field(field), n, lo, hi, iso)
    got = (v.numpy(), t.numpy().astype(np.uint32))
    if n != (1, 1, 1):
        assert len(want[1]) > 0
    assert_identical(got, want)


def test_sparse_extract_without_a_gpu_fails_with_no_device(hp):
    if hp.device_count() > 0:
        pytest.skip("a GPU is present")
    L = hp.lib()
    nv, nt, pv, pt = C.c_size_t(), C.c_size_t(), C.c_void_p(), C.c_void_p()
    res = (C.c_uint32 * 3)(16, 16, 16)
    assert L.hpsdf_extract_isosurface_sparse(None, res, None, None, 0.0, C.byref(nv), C.byref(pv), C.byref(nt), C.byref(pt)) == hp.ERR_NO_DEVICE
    with pytest.raises(hp.HpsdfError) as e:
        hp.Octree().ExtractIsosurfaceSparse(16)
    assert e.value.status == hp.ERR_NO_DEVICE


def test_facade_extract_isosurface_sparse_compiles_without_a_gpu(tmp_path):
    src = tmp_path / "t.cpp"
    src.write_text('#include "hpsdf.hpp"\nint main() { SDF::Octree t; std::vector<float> v; std::vector<uint32_t> i; const uint32_t r[3] = { 8, 8, 8 };\n'
                   'try { t.ExtractIsosurfaceSparse(r, 0.0, v, i); } catch (const SDF::Error& e) { return e.status == HPSDF_ERR_INVALID_ARG ? 0 : 1; } return 2; }\n')
    exe = str(tmp_path / "t")
    subprocess.check_call([GXX, "-std=c++17", "-I", os.path.join(ROOT, "include"), str(src), "-L", os.path.join(PKG, "lib"), "-lhpsdf", "-o", exe])
    assert subprocess.run([exe], env=dict(os.environ, LD_LIBRARY_PATH=os.path.join(PKG, "lib"))).returncode == 0


# ---- GPU -----------------------------------------------------------------------------------------------------------------

NAMES = ["custom_domain", "c2_csg", "sphere_poly_1e8"]


@pytest.fixture(scope="module")
def trees(hp):
    out = {}
    for name in NAMES:
        cfg, prog = product_cfg(hp, name)
        t = hp.Octree()
        t.Create(cfg, prog)
        out[name] = t
    return out


@pytest.fixture(scope="module")
def c3(hp):
    from meshgen import bumpy_torus, mesh_root
    verts, tris = bumpy_torus(1000, 435)
    lo, hi = mesh_root(verts)
    tree = hp.Octree()
    tree.Create(hp.Config(target_error_threshold=1e-6, nearness_type=0, nearness_strength=0.0, continuity_enforce=1, continuity_strength=8.0,
                          root_min=lo, root_max=hi), hp.SdfProgram([("mesh", [], hp.Mesh(verts, tris))]), hp.BuildOpts(max_degree=11))
    return tree, np.asarray(lo, np.float32).astype(np.float64), np.asarray(hi, np.float32).astype(np.float64)


def sub_box(name):
    lo, hi = root_box(name)
    size = hi - lo
    return lo + 0.1 * size, hi + np.array([0.15, 0.1, -0.05]) * size       # past the root on +x and +y: DBL_MAX corners


def checker_mesh(tree, n, lo, hi, iso):
    return R.extract(tree.Query(R.grid_points(n, lo, hi)), n, lo, hi, iso)


def box_of(name, sub):
    return sub_box(name) if sub else root_box(name)


SMALL = [(40, 48, 56), (15, 16, 17), (16, 16, 16), (33, 1, 47), (1, 1, 1), (1024, 3, 700)]
# an axis above 1024 cells: the sparse pipeline at any size; partial last blocks of 12, 2 and 1 cells, an exact multiple of
# 16, one-cell and two-cell axes
FORCED_SPARSE = [(1030, 48, 56), (1025, 1, 17), (2048, 16, 33)]


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("n", SMALL + FORCED_SPARSE)
@pytest.mark.parametrize("iso_frac", [0.0, 0.02])
@pytest.mark.parametrize("sub", [False, True])
def test_same_bits_as_the_checker(trees, name, n, iso_frac, sub):
    lo, hi = box_of(name, sub)
    iso = iso_frac * float(root_box(name)[1][0] - root_box(name)[0][0])
    b = (lo, hi) if sub else None
    want = checker_mesh(trees[name], n, lo, hi, iso)
    if n in ((40, 48, 56), (1030, 48, 56)):
        assert len(want[1]) > 0
    got = trees[name].ExtractIsosurfaceSparse(n, iso, b)
    assert_identical(got, want)
    if max(n) <= 1024:
        assert_identical(trees[name].ExtractIsosurface(n, iso, b), got)


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("iso", [-10.0, 10.0, np.inf, -np.inf, np.nan])
def test_empty_and_full_grids(trees, name, iso):
    for sub in (False, True):
        lo, hi = box_of(name, sub)
        b = (lo, hi) if sub else None
        for n in ((40, 48, 56), (1030, 48, 56)):
            got = trees[name].ExtractIsosurfaceSparse(n, iso, b)
            if not sub:                          # the sub-box reaches past the root, where DBL_MAX corners are outside
                assert len(got[0]) == 0 and len(got[1]) == 0
            assert_identical(got, checker_mesh(trees[name], n, lo, hi, iso))


@pytest.mark.gpu
@pytest.mark.parametrize("iso", [np.inf, -np.inf, np.nan])
def test_no_crossing_at_16384_is_certified_at_the_top_level(trees, iso):
    """No grid point is inside (iso = -inf, NaN) or all are (+inf): the top level certifies every block, so the largest grid
    takes no more scratch than a small one."""
    v, t = trees["c2_csg"].ExtractIsosurfaceSparse(16384, iso)
    assert len(v) == 0 and len(t) == 0


@pytest.mark.gpu
def test_c3_at_1024_equals_the_slab_checker(c3):
    tree, lo, hi = c3
    got = tree.ExtractIsosurfaceSparse(1024)
    assert len(got[1]) > 10 ** 7
    assert_identical(tree.ExtractIsosurface(1024), got)
    assert_equals_slab(got, slab_mesh(tree, (1024,) * 3, lo, hi, 0.0))


@pytest.mark.gpu
def test_iso_at_grid_values_and_block_bounds(hp, trees):
    """Leaves of every degree 0-12 with random coefficients. iso is Query's value at grid points (t = 1 vertices), and the
    certified f_lo and f_hi of the grid's own 16³ blocks (boxes with the grid's corner coordinates), so that the culling
    comparisons f_lo >= iso and f_hi < iso meet equality."""
    from test_gpu_derivatives import every_degree_block
    tree = hp.Octree()
    tree.FromMemoryBlock(hp.MemoryBlock.frombytes(every_degree_block(hp, trees["c2_csg"].ToMemoryBlockBytes())))
    lo, hi = root_box("c2_csg")
    rng = np.random.default_rng(3)
    n = (1030, 40, 33)
    P = R.grid_points(n, lo, hi)
    vals = tree.Query(P)
    axes = R.grid_axes(n, lo, hi)
    nb = [(x + 15) // 16 for x in n]
    bi, bj, bk = (np.arange(c) for c in nb)
    B = np.stack(np.meshgrid(bi, bj, bk, indexing="ij"), -1).reshape(-1, 3)
    blo = np.stack([axes[a][16 * B[:, a]] for a in range(3)], 1)
    bhi = np.stack([axes[a][np.minimum(16 * B[:, a] + 16, n[a])] for a in range(3)], 1)
    f_lo, f_hi = tree.QueryBounds(blo, bhi)
    finite = np.nonzero(f_hi < np.finfo(np.float64).max)[0]
    pick = rng.choice(finite, 4, replace=False)
    isos = np.concatenate([vals[rng.choice(len(P), 4, replace=False)], f_lo[pick], f_hi[pick]])
    for iso in isos:
        want = R.extract(vals, n, lo, hi, float(iso))
        assert_identical(tree.ExtractIsosurfaceSparse(n, float(iso)), want)


def slab_mesh(tree, n, lo, hi, iso):
    import torch
    v, t = S.extract(S.query_field(tree), n, lo, hi, iso, device="cuda")
    return v, t


def assert_equals_slab(got, want):
    import torch
    gv, gt = got
    wv, wt = want
    assert gv.shape == tuple(wv.shape) and gt.shape == tuple(wt.shape)
    assert torch.equal(torch.from_numpy(gv.view(np.int32)).cuda(), wv.view(torch.int32))
    assert torch.equal(torch.from_numpy(gt.astype(np.int64)).cuda(), wt)


@pytest.mark.gpu
def test_beyond_1024_equals_the_slab_checker(trees):
    name = "sphere_poly_1e8"
    lo, hi = root_box(name)
    n = (2048, 1100, 1536)
    got = trees[name].ExtractIsosurfaceSparse(n, 0.0)
    assert len(got[1]) > 10 ** 6
    assert_equals_slab(got, slab_mesh(trees[name], n, lo, hi, 0.0))
    n = (16384, 2, 900)
    got = trees[name].ExtractIsosurfaceSparse(n, 0.0)
    assert_equals_slab(got, slab_mesh(trees[name], n, lo, hi, 0.0))
    n, clo, chi = (4000, 4097, 1), np.array([0.5, 0.5, 1.9]), np.array([3.5, 3.5, 2.1])     # both z-planes cut the sphere
    got = trees["custom_domain"].ExtractIsosurfaceSparse(n, 0.0, (clo, chi))
    assert len(got[1]) > 0
    assert_equals_slab(got, slab_mesh(trees["custom_domain"], n, clo, chi, 0.0))
    blo, bhi = sub_box("c2_csg")
    n = (1500, 2049, 1030)
    got = trees["c2_csg"].ExtractIsosurfaceSparse(n, 0.01, (blo, bhi))
    assert len(got[1]) > 10 ** 6
    assert_equals_slab(got, slab_mesh(trees["c2_csg"], n, blo, bhi, 0.01))


def closed_oriented_all_used(v, t):
    """isosurface_ref.mesh_report's closed_oriented and all_used, in torch on the GPU for meshes of 10^8 triangles."""
    import torch
    T = torch.from_numpy(t.astype(np.int64)).cuda()
    nv = len(v)
    a, b = T.reshape(-1), T[:, [1, 2, 0]].reshape(-1)
    key, _ = torch.sort(a * nv + b)
    once = bool((key[1:] != key[:-1]).all())
    rev = b * nv + a
    pos = torch.searchsorted(key, rev).clamp(max=len(key) - 1)
    paired = bool((key[pos] == rev).all())
    used = torch.zeros(nv, dtype=torch.bool, device="cuda")
    used[a] = True
    return once and paired, bool(used.all())


@pytest.mark.gpu
def test_c3_at_4096_is_a_closed_surface_on_the_tree(hp, c3):
    """1.2 TB of dense scratch; the slab checker would need several minutes here, so the bit check stays at the 2048-class
    sizes above."""
    tree, lo, hi = c3
    n = 4096
    v, t = tree.ExtractIsosurfaceSparse(n)
    print("C3 at 4096^3: %d vertices, %d triangles" % (len(v), len(t)))
    assert len(t) > 10 ** 8
    closed, used = closed_oriented_all_used(v, t)
    assert closed and used
    diag = np.linalg.norm((hi - lo) / n)
    sample = v[np.random.default_rng(9).choice(len(v), 10000, replace=False)].astype(np.float64)
    # a vertex lies on a grid edge across which Query changes sign. On this sample the median |Query| is 1e-7; 65 of the 10^4
    # vertices lie beyond 2 cell diagonals (0.44e-3), the largest at 4.0e-3. Their cause is not established (DESIGN §15)
    q = np.abs(tree.Query(sample))
    assert np.median(q) <= 2 * diag and q.max() <= 0.01
    hp.Mesh(v, t)


@pytest.mark.gpu
def test_determinism_across_reruns_clones_and_memory_blocks(hp, trees):
    tree = trees["c2_csg"]
    n, iso = (33, 40, 1047), 0.01                 # an axis above 1024: the sparse pipeline
    first = tree.ExtractIsosurfaceSparse(n, iso)
    assert len(first[1]) > 0
    assert_identical(tree.ExtractIsosurfaceSparse(n, iso), first)
    assert_identical(tree.copy().ExtractIsosurfaceSparse(n, iso), first)
    copy = hp.Octree()
    copy.FromMemoryBlock(hp.MemoryBlock.frombytes(tree.ToMemoryBlockBytes()))
    assert_identical(copy.ExtractIsosurfaceSparse(n, iso), first)         # its first call builds the bounds table
    assert_identical(copy.ExtractIsosurfaceSparse(n, iso), first)


@pytest.mark.gpu
def test_empty_result_and_argument_errors(hp, trees):
    tree = trees["c2_csg"]
    L = hp.lib()
    fn = L.hpsdf_extract_isosurface_sparse
    nv, nt, pv, pt = C.c_size_t(7), C.c_size_t(7), C.c_void_p(1), C.c_void_p(1)
    res = (C.c_uint32 * 3)(32, 32, 32)
    assert fn(tree._h, res, None, None, -10.0, C.byref(nv), C.byref(pv), C.byref(nt), C.byref(pt)) == hp.OK
    assert nv.value == 0 and nt.value == 0 and pv.value is None and pt.value is None
    v, t = tree.ExtractIsosurfaceSparse(32, -10.0)
    assert v.shape == (0, 3) and t.shape == (0, 3)
    lo, hi = root_box("c2_csg")
    for bad in (0, 16385, (16, 0, 16), (16, 16, 16385), (2 ** 32 - 1, 16, 16)):
        with pytest.raises(hp.HpsdfError) as e:
            tree.ExtractIsosurfaceSparse(bad)
        assert e.value.status == hp.ERR_INVALID_ARG
    for box in ((hi, lo), ((lo[0], lo[1], hi[2]), (hi[0], hi[1], hi[2])), ((lo[0], np.nan, lo[2]), hi), (lo, (hi[0], np.inf, hi[2]))):
        with pytest.raises(hp.HpsdfError) as e:
            tree.ExtractIsosurfaceSparse(16, 0.0, box)
        assert e.value.status == hp.ERR_INVALID_ARG
    dlo = (C.c_double * 3)(*lo)
    for a, b in ((dlo, None), (None, dlo)):
        assert fn(tree._h, res, a, b, 0.0, C.byref(nv), C.byref(pv), C.byref(nt), C.byref(pt)) == hp.ERR_INVALID_ARG
    assert fn(None, res, None, None, 0.0, C.byref(nv), C.byref(pv), C.byref(nt), C.byref(pt)) == hp.ERR_INVALID_ARG
    assert fn(tree._h, None, None, None, 0.0, C.byref(nv), C.byref(pv), C.byref(nt), C.byref(pt)) == hp.ERR_INVALID_ARG
    assert fn(tree._h, res, None, None, 0.0, None, C.byref(pv), C.byref(nt), C.byref(pt)) == hp.ERR_INVALID_ARG


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
    const uint32_t res[3] = { 24, 1100, 40 };
    std::vector<float> v;
    std::vector<uint32_t> t;
    tree.ExtractIsosurfaceSparse(res, 0.0, v, t);
    const double lo[3] = { -0.2, -0.45, -0.4 }, hi[3] = { 0.5, 0.4, 0.45 };
    std::vector<float> v2;
    std::vector<uint32_t> t2;
    tree.ExtractIsosurfaceSparse(res, 0.01, v2, t2, lo, hi);
    MemoryBlock b = tree.ToMemoryBlock();
    FILE* f = std::fopen(argv[1], "wb");
    const size_t counts[5] = { v.size() / 3, t.size() / 3, v2.size() / 3, t2.size() / 3, b.size };
    std::fwrite(counts, sizeof(counts), 1, f);
    std::fwrite(v.data(), 4, v.size(), f); std::fwrite(t.data(), 4, t.size(), f);
    std::fwrite(v2.data(), 4, v2.size(), f); std::fwrite(t2.data(), 4, t2.size(), f);
    std::fwrite(b.ptr, 1, b.size, f);
    std::fclose(f);
    std::free(b.ptr);
    return 0;
}
"""


@pytest.mark.gpu
def test_cpp_facade_matches_the_python_call(hp, tmp_path):
    src, exe, dump = tmp_path / "iso.cpp", str(tmp_path / "iso"), str(tmp_path / "iso.bin")
    src.write_text(FACADE_SRC)
    subprocess.check_call([GXX, "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), str(src), "-L", os.path.join(PKG, "lib"), "-lhpsdf", "-o", exe])
    env = dict(os.environ, LD_LIBRARY_PATH=os.path.join(PKG, "lib") + ":" + os.environ.get("LD_LIBRARY_PATH", ""))
    out = subprocess.run([exe, dump], env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    raw = open(dump, "rb").read()
    counts = np.frombuffer(raw[:40], np.uint64).astype(np.int64)
    off, parts = 40, []
    for k, dt in zip(counts[:4], (np.float32, np.uint32, np.float32, np.uint32)):
        parts.append(np.frombuffer(raw[off:off + 12 * k], dt).reshape(-1, 3))
        off += 12 * k
    tree = hp.Octree()
    tree.FromMemoryBlock(hp.MemoryBlock.frombytes(raw[off:off + counts[4]]))
    v, t = tree.ExtractIsosurfaceSparse((24, 1100, 40))
    assert len(t) and np.array_equal(parts[0], v) and np.array_equal(parts[1], t)
    v2, t2 = tree.ExtractIsosurfaceSparse((24, 1100, 40), 0.01, ((-0.2, -0.45, -0.4), (0.5, 0.4, 0.45)))
    assert len(t2) and np.array_equal(parts[2], v2) and np.array_equal(parts[3], t2)
