"""hpsdf_extract_isosurface / Octree.ExtractIsosurface: marching tetrahedra over a grid of Query values, checked bit for bit
against the numpy restatement of the contract (isosurface_ref.py), and as a mesh: closed, oriented, of the right genus and
volume, accepted by hp.Mesh, close to the source surface."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import isosurface_ref as R
from cases import CASES, root_points
from common import product_cfg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "hp-adaptive-signed-distance-field-octree_b200")
GXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"


def root_box(name):
    k = CASES[name]["cfg"]
    lo = np.asarray(k.get("root_min", (-0.5,) * 3), np.float32).astype(np.float64)
    hi = np.asarray(k.get("root_max", (0.5,) * 3), np.float32).astype(np.float64)
    return lo, hi


def checker_mesh(tree, n, lo, hi, iso):
    return R.extract(tree.Query(R.grid_points(n, lo, hi)), n, lo, hi, iso)


def assert_same_mesh(got, want):
    (gv, gt), (wv, wt) = got, want
    assert gv.dtype == np.float32 and gt.dtype == np.uint32
    assert gv.shape == wv.shape and gt.shape == wt.shape
    assert np.array_equal(gv, wv)
    assert np.array_equal(R.canonical_rows(gt), R.canonical_rows(wt))


# ---- CPU: the checker itself, and the entry point without a device -------------------------------------------------------

def sphere_field(P, r=0.31):
    return np.sqrt((P ** 2).sum(1)) - r


def test_checker_gives_a_closed_sphere_of_the_right_volume():
    n, lo, hi, r = (64, 64, 64), (-0.5,) * 3, (0.5,) * 3, 0.31
    v, t = R.extract(sphere_field(R.grid_points(n, lo, hi), r), n, lo, hi, 0.0)
    rep = R.mesh_report(v, t)
    assert rep["closed_oriented"] and rep["all_used"] and rep["euler"] == 2
    exact = 4.0 / 3.0 * np.pi * r ** 3
    assert rep["volume"] > 0 and abs(rep["volume"] - exact) <= 0.02 * exact


def test_checker_gives_a_torus_of_genus_one():
    n, lo, hi = (48, 40, 32), (-0.5,) * 3, (0.5,) * 3
    P = R.grid_points(n, lo, hi)
    f = np.sqrt((np.sqrt(P[:, 0] ** 2 + P[:, 1] ** 2) - 0.3) ** 2 + P[:, 2] ** 2) - 0.1
    rep = R.mesh_report(*R.extract(f, n, lo, hi, 0.0))
    assert rep["closed_oriented"] and rep["all_used"] and rep["euler"] == 0 and rep["volume"] > 0


def test_checker_winding_flips_with_the_sign_of_the_field():
    n, lo, hi = (20, 24, 28), (-0.5,) * 3, (0.5,) * 3
    f = sphere_field(R.grid_points(n, lo, hi), 0.3071)
    _, t = R.extract(f, n, lo, hi, 0.0)
    v2, t2 = R.extract(-f, n, lo, hi, 0.0)               # the same crossings, inside and outside swapped
    assert R.mesh_report(v2, t2)["volume"] < 0 and len(t2) == len(t)


def test_extract_without_a_gpu_fails_with_no_device(hp):
    if hp.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(hp.HpsdfError) as e:
        hp.Octree().ExtractIsosurface(16)
    assert e.value.status == hp.ERR_NO_DEVICE


def test_facade_extract_isosurface_compiles_without_a_gpu(tmp_path):
    src = tmp_path / "t.cpp"
    src.write_text('#include "hpsdf.hpp"\nint main() { SDF::Octree t; std::vector<float> v; std::vector<uint32_t> i; const uint32_t r[3] = { 8, 8, 8 };\n'
                   'try { t.ExtractIsosurface(r, 0.0, v, i); } catch (const SDF::Error& e) { return e.status == HPSDF_ERR_INVALID_ARG ? 0 : 1; } return 2; }\n')
    exe = str(tmp_path / "t")
    subprocess.check_call([GXX, "-std=c++17", "-I", os.path.join(ROOT, "include"), str(src), "-L", os.path.join(PKG, "lib"), "-lhpsdf", "-o", exe])
    assert subprocess.run([exe], env=dict(os.environ, LD_LIBRARY_PATH=os.path.join(PKG, "lib"))).returncode == 0


# ---- GPU -----------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def trees(hp):
    out = {}
    for name in ("custom_domain", "c2_csg", "sphere_poly_1e8"):
        cfg, prog = product_cfg(hp, name)
        t = hp.Octree()
        t.Create(cfg, prog)
        out[name] = t
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["custom_domain", "c2_csg", "sphere_poly_1e8"])
@pytest.mark.parametrize("iso_frac", [0.0, 0.02])
@pytest.mark.parametrize("sub_box", [False, True])
def test_bit_exact_against_the_checker(trees, name, iso_frac, sub_box):
    n = (40, 48, 56)
    lo, hi = root_box(name)
    size = hi - lo
    iso = iso_frac * float(size[0])
    if sub_box:                                  # past the root on the +x and +y faces: DBL_MAX corners there
        lo, hi = lo + 0.1 * size, hi + np.array([0.15, 0.1, -0.05]) * size
        got = trees[name].ExtractIsosurface(n, iso, (lo, hi))
    else:
        got = trees[name].ExtractIsosurface(n, iso)
    want = checker_mesh(trees[name], n, lo, hi, iso)
    assert len(want[1]) > 0
    assert_same_mesh(got, want)


@pytest.mark.gpu
def test_sphere_in_a_custom_domain_is_closed_and_accurate(hp, trees):
    v, t = trees["custom_domain"].ExtractIsosurface(128)
    hp.Mesh(v, t)
    rep = R.mesh_report(v, t)
    assert rep["closed_oriented"] and rep["all_used"] and rep["euler"] == 2
    exact = 4.0 / 3.0 * np.pi * 0.75 ** 3
    assert abs(rep["volume"] - exact) <= 0.02 * exact
    assert np.abs(np.linalg.norm(v.astype(np.float64) - 2.0, axis=1) - 0.75).max() <= 0.01


@pytest.mark.gpu
def test_csg_mesh_has_the_sign_of_the_tree(hp, trees):
    tree, n = trees["c2_csg"], 128
    v, t = tree.ExtractIsosurface(n)
    mesh = hp.Mesh(v, t)
    assert R.mesh_report(v, t)["closed_oriented"]
    lo, hi = root_box("c2_csg")
    diag = np.linalg.norm((hi - lo) / n)
    pts = root_points(CASES["c2_csg"]["cfg"], 60000, seed=11)
    q = tree.Query(pts)
    far = np.abs(q) > 2 * diag
    pts, q = pts[far][:20000], q[far][:20000]
    assert len(q) == 20000
    assert np.array_equal(mesh.SignedDistanceAtPt(pts) > 0, q > 0)


@pytest.mark.gpu
def test_surface_leaving_the_root_gives_an_open_mesh(hp, trees):
    v, t = trees["sphere_poly_1e8"].ExtractIsosurface(64)
    assert len(t) and not R.mesh_report(v, t)["closed_oriented"]
    with pytest.raises(hp.HpsdfError) as e:
        hp.Mesh(v, t)
    assert e.value.status == hp.ERR_MESH


@pytest.mark.gpu
def test_mesh_octree_mesh_round_trip(hp):
    from meshgen import bumpy_torus, mesh_root
    verts, tris = bumpy_torus(200, 90)
    lo, hi = mesh_root(verts)
    src = hp.Mesh(verts, tris)
    tree = hp.Octree()
    tree.Create(hp.Config(target_error_threshold=1e-6, continuity_enforce=0, root_min=lo, root_max=hi), hp.SdfProgram([("mesh", [], src)]))
    n = 160
    v, t = tree.ExtractIsosurface(n)
    box_lo, box_hi = np.asarray(lo, np.float32).astype(np.float64), np.asarray(hi, np.float32).astype(np.float64)
    assert_same_mesh((v, t), checker_mesh(tree, (n, n, n), box_lo, box_hi, 0.0))
    rep = R.mesh_report(v, t)
    print("round trip: %d vertices, %d triangles, V - E + F = %d" % (len(v), len(t), rep["euler"]))
    assert rep["closed_oriented"] and rep["all_used"]
    out = hp.Mesh(v, t)
    diag = np.linalg.norm((box_hi - box_lo) / n)
    pts = np.random.default_rng(5).uniform(box_lo, box_hi, (20000, 3)).astype(np.float32)
    # the tree's field departs from the mesh's by up to 0.048 (7 cells) in a few places, where its zero set carries small extra
    # closed components (DESIGN §11): V - E + F is the tree's, not a torus's, and the distances agree to a few cell diagonals
    diff = np.abs(out.SignedDistanceAtPt(pts).astype(np.float64) - src.SignedDistanceAtPt(pts))
    assert diff.max() <= 4 * diag, diff.max()


@pytest.mark.gpu
def test_empty_result_and_argument_errors(hp, trees):
    tree = trees["c2_csg"]
    L = hp.lib()
    nv, nt, pv, pt = C.c_size_t(7), C.c_size_t(7), C.c_void_p(1), C.c_void_p(1)
    res = (C.c_uint32 * 3)(32, 32, 32)
    assert L.hpsdf_extract_isosurface(tree._h, res, None, None, -10.0, C.byref(nv), C.byref(pv), C.byref(nt), C.byref(pt)) == hp.OK
    assert nv.value == 0 and nt.value == 0 and pv.value is None and pt.value is None
    v, t = tree.ExtractIsosurface(32, -10.0)
    assert v.shape == (0, 3) and t.shape == (0, 3)
    lo, hi = root_box("c2_csg")
    for bad in (0, 1025, (16, 0, 16), (16, 16, 1025)):
        with pytest.raises(hp.HpsdfError) as e:
            tree.ExtractIsosurface(bad)
        assert e.value.status == hp.ERR_INVALID_ARG
    for box in ((hi, lo), ((lo[0], lo[1], hi[2]), (hi[0], hi[1], hi[2]))):
        with pytest.raises(hp.HpsdfError) as e:
            tree.ExtractIsosurface(16, 0.0, box)
        assert e.value.status == hp.ERR_INVALID_ARG
    dlo = (C.c_double * 3)(*lo)
    for a, b in ((dlo, None), (None, dlo)):
        assert L.hpsdf_extract_isosurface(tree._h, res, a, b, 0.0, C.byref(nv), C.byref(pv), C.byref(nt), C.byref(pt)) == hp.ERR_INVALID_ARG
    assert L.hpsdf_extract_isosurface(None, res, None, None, 0.0, C.byref(nv), C.byref(pv), C.byref(nt), C.byref(pt)) == hp.ERR_INVALID_ARG
    assert L.hpsdf_extract_isosurface(tree._h, None, None, None, 0.0, C.byref(nv), C.byref(pv), C.byref(nt), C.byref(pt)) == hp.ERR_INVALID_ARG


@pytest.mark.gpu
def test_tree_from_a_memory_block_gives_the_same_mesh(hp, trees):
    tree = trees["c2_csg"]
    copy = hp.Octree()
    mb = tree.ToMemoryBlock()
    try:
        copy.FromMemoryBlock(mb)
    finally:
        mb.free()
    assert_same_mesh(copy.ExtractIsosurface((33, 40, 47), 0.01), tree.ExtractIsosurface((33, 40, 47), 0.01))


@pytest.mark.gpu
def test_c3_tree_at_full_resolution(hp):
    from meshgen import bumpy_torus, mesh_root
    verts, tris = bumpy_torus(1000, 435)
    lo, hi = mesh_root(verts)
    src = hp.Mesh(verts, tris)
    tree = hp.Octree()
    tree.Create(hp.Config(target_error_threshold=1e-6, nearness_type=0, nearness_strength=0.0, continuity_enforce=1, continuity_strength=8.0,
                          root_min=lo, root_max=hi), hp.SdfProgram([("mesh", [], src)]), hp.BuildOpts(max_degree=11))
    n = 1024
    v, t = tree.ExtractIsosurface(n)
    hp.Mesh(v, t)
    rep = R.mesh_report(v, t)
    print("C3 at 1024^3: %d vertices, %d triangles, V - E + F = %d" % (len(v), len(t), rep["euler"]))
    assert rep["closed_oriented"] and rep["all_used"]
    box_lo, box_hi = np.asarray(lo, np.float32).astype(np.float64), np.asarray(hi, np.float32).astype(np.float64)
    diag = np.linalg.norm((box_hi - box_lo) / n)
    sample = v[np.random.default_rng(9).choice(len(v), 10000, replace=False)].astype(np.float64)
    # each vertex lies on a grid edge (at most one cell diagonal long) across which Query changes sign; the tree's field is
    # piecewise polynomial, with small jumps across leaf faces and a gradient that is not exactly 1, hence the factor 2
    assert np.abs(tree.Query(sample)).max() <= 2 * diag


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
    const uint32_t res[3] = { 24, 32, 40 };
    std::vector<float> v;
    std::vector<uint32_t> t;
    tree.ExtractIsosurface(res, 0.0, v, t);
    const double lo[3] = { -0.2, -0.45, -0.4 }, hi[3] = { 0.5, 0.4, 0.45 };
    std::vector<float> v2;
    std::vector<uint32_t> t2;
    tree.ExtractIsosurface(res, 0.01, v2, t2, lo, hi);
    MemoryBlock b = tree.ToMemoryBlock();
    FILE* f = std::fopen(argv[1], "wb");
    const size_t counts[5] = { v.size() / 3, t.size() / 3, v2.size() / 3, t2.size() / 3, b.size };
    std::fwrite(counts, sizeof(counts), 1, f);
    std::fwrite(v.data(), 4, v.size(), f); std::fwrite(t.data(), 4, t.size(), f);
    std::fwrite(v2.data(), 4, v2.size(), f); std::fwrite(t2.data(), 4, t2.size(), f);
    std::fwrite(b.ptr, 1, b.size, f);
    std::fclose(f);
    std::free(b.ptr);
    std::printf("%zu %zu %zu %zu\n", counts[0], counts[1], counts[2], counts[3]);
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
    v, t = tree.ExtractIsosurface((24, 32, 40))
    assert len(t) and np.array_equal(parts[0], v) and np.array_equal(parts[1], t)
    v2, t2 = tree.ExtractIsosurface((24, 32, 40), 0.01, ((-0.2, -0.45, -0.4), (0.5, 0.4, 0.45)))
    assert len(t2) and np.array_equal(parts[2], v2) and np.array_equal(parts[3], t2)
