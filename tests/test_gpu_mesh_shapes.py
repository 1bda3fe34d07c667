"""GPU: the device mesh signed distance on sharp, thin, high-valence, nested and non-manifold shapes, against the oracle bit
for bit and against exact geometry.

Bit identity alone cannot catch an error that the oracle shares, and the device-against-device tests of
test_gpu_mesh_wide.py cannot catch an error in the set-up both walks share (half-edges, pseudonormals, BVH, oriented
boxes). The exact check (mesh_exact.py, bound K of test_mesh_exact.py) does: a triangle lost by pruning or a box that
misses its triangles moves the distance by far more than K ulps."""
import numpy as np
import pytest

from common import rel_inf
from meshgen import SHAPES, mesh_root, point_sets
from test_gpu_parity import compare_with_oracle_tree
from test_mesh_exact import check_against_exact, exact_shape, format_report, pairing_meshes

pytestmark = pytest.mark.gpu


def bits(x):
    return np.ascontiguousarray(x, np.float32).view(np.uint32)


@pytest.mark.parametrize("name", list(SHAPES))
def test_distance_is_bit_identical_to_the_oracle(hp, oracle, name):
    """At the shape's own scale and at the scale of the exact check: every point class, as uint32 bits (so -0.0 on a
    vertex counts), against the oracle's BVH walk and its brute-force loop; and the mesh bounds against numpy's."""
    counts = []
    for v, t in (SHAPES[name](), exact_shape(name)[:2]):
        m, om = hp.Mesh(v, t), oracle.OracleMesh(v, t)
        n = 0
        for cls, p in point_sets(v, t, np.random.default_rng(sum(map(ord, name)))).items():
            d = bits(m.SignedDistanceAtPt(p))
            for use_bvh in (True, False):
                o = bits(om.sdf(p, use_bvh, 8))
                bad = np.flatnonzero(d != o)
                assert len(bad) == 0, "%s/%s (%s): %d of %d differ, first %s: device %r oracle %r" % (
                    name, cls, "bvh" if use_bvh else "brute force", len(bad), len(p), p[bad[0]].tolist(),
                    d[bad[0]:bad[0] + 1].view(np.float32)[0], o[bad[0]:bad[0] + 1].view(np.float32)[0])
            n += len(p)
        mn, mx = m.CalculateMeshAABB()
        assert np.array_equal(mn, v.min(0)) and np.array_equal(mx, v.max(0))
        counts.append(n)
        m.close()
        om.close()
    print("%s: %s points bit-identical" % (name, " + ".join(map(str, counts))))


@pytest.mark.parametrize("name", list(SHAPES))
def test_distance_matches_exact_geometry(hp, name):
    v, t, s = exact_shape(name)
    m = hp.Mesh(v, t)
    sets = point_sets(v, t, np.random.default_rng(sum(map(ord, name))))
    report = check_against_exact(name, v, t, sets, m.SignedDistanceAtPt)
    print("%s (x%g): worst |d - exact| / u(|p| + |v|): %s" % (name, s, format_report(report)))
    m.close()


def straddling_cells(v, depth_count=9):
    """One cell per depth 0..8 of the root box mesh_root(v), containing a corner of the cube at even depths and an edge
    midpoint at odd depths: (root min, root max, cells (n, 4) f32 as unit-cube centre and half size, depths)."""
    lo, hi = (np.array(x) for x in mesh_root(v))
    h = float(v.max())
    targets = [np.array([h, h, h]), np.array([h, 0.1 * h, -h])]
    cells, depths = [], []
    for depth in range(depth_count):
        u = (targets[depth % 2] - (lo + hi) / 2) / (hi - lo)
        half = 0.5 ** (depth + 1)
        idx = np.floor((u + 0.5) / (2 * half))
        cells.append(np.concatenate([(idx + 0.5) * 2 * half - 0.5, [half]]))
        depths.append(depth)
    return lo, hi, np.array(cells, np.float32), np.array(depths)


@pytest.mark.parametrize("degree", list(range(1, 12)))
def test_fits_on_cells_straddling_edges_and_corners(hp, oracle, degree):
    """Every fit degree at depths 0..8 on the cube, whose edges and corners make the SDF non-smooth in every such cell.
    The single-mesh program takes meshSampleKernel with the per-fit cut; [mesh, sphere, union] takes sampleKernel."""
    from oracle import hpref
    v, t = SHAPES["cube"]()
    m, om = hp.Mesh(v, t), oracle.OracleMesh(v, t)
    lo, hi, cells, depths = straddling_cells(v)
    cfg = hp.Config(target_error_threshold=1e-6, continuity_enforce=0, root_min=tuple(lo), root_max=tuple(hi))
    ocfg = hpref.make_config(threshold=1e-6, continuity=False, root_min=tuple(lo), root_max=tuple(hi), threads=1)
    for extra in ([], [("sphere", [0.1, 0.05, 0.0, 0.3]), ("union", [])]):
        coeffs, err, _ = hp.fit_batch(cfg, hp.SdfProgram([("mesh", [], m)] + extra), cells, depths, degree)
        oprog = hpref.make_program([("mesh", [], om.h)] + extra)
        for i, depth in enumerate(depths):
            c0, half = cells[i, :3].astype(np.float64), float(cells[i, 3])
            c, e = oracle.oracle_fit(ocfg, oprog, c0 - half, c0 + half, degree, int(depth))
            assert rel_inf(coeffs[i], c) <= 1e-10, (len(extra), depth, rel_inf(coeffs[i], c))
            # err is the energy of the n top-shell coefficients: if each is off by at most eta = 1e-12 |c|inf (rounding of
            # the sample sums), the sum of their squares is off by at most 2 eta sqrt(n err) + n eta^2
            eta, n_top = 1e-12 * np.abs(c).max(), (degree + 1) * (degree + 2) // 2
            assert abs(err[i] - e) <= 1e-9 * e + 2 * eta * np.sqrt(n_top * e) + n_top * eta ** 2, (len(extra), depth, err[i], e)


@pytest.mark.parametrize("name", ["cube", "star_prism", "thin_plate"])
def test_build_matches_the_oracle_tree(hp, oracle, name):
    from oracle import hpref
    v, t = SHAPES[name]()
    m, om = hp.Mesh(v, t), oracle.OracleMesh(v, t)
    lo, hi = mesh_root(v)
    kw = dict(threshold=1e-5, continuity=False, root_min=lo, root_max=hi)
    o = oracle.OracleTree.build(hpref.make_config(threads=8, **kw), hpref.make_program([("mesh", [], om.h)]), threads=8)
    tree = hp.Octree()
    tree.Create(hp.Config(target_error_threshold=1e-5, continuity_enforce=0, root_min=lo, root_max=hi), hp.SdfProgram([("mesh", [], m)]))
    worst, div = compare_with_oracle_tree(hp, tree, o, kw)
    print("%s tree: %d nodes, worst coefficient error %.2g, %d divergent cells" % (name, tree.stats()["n_nodes"], worst, div))


def test_bad_meshes_are_rejected(hp):
    """mesh.cpp reads the pairing flags before any kernel reads the half-edges, so these are safe to create."""
    for name, (v, t, accepted) in pairing_meshes().items():
        if accepted:
            hp.Mesh(v, t).close()
            continue
        with pytest.raises(hp.HpsdfError) as e:
            hp.Mesh(v, t)
        assert e.value.status == hp.ERR_MESH, name
    v, t = SHAPES["cube"]()
    bad = t.copy()
    bad[5, 1] = len(v)
    with pytest.raises(hp.HpsdfError) as e:
        hp.Mesh(v, bad)
    assert e.value.status == hp.ERR_INVALID_ARG
