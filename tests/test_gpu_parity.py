"""GPU: the CUDA path through the C ABI against the CPU oracle and the golden vectors from the reference.

Tolerances are BASELINE.json's: identical topology, per-leaf |dc|inf/|c|inf <= 1e-10, |dQuery| <= 1e-9.
"""
import numpy as np
import pytest

from cases import CASES, root_points, leaf_table, path_code, cell_of, divergent_cells
from common import golden, oracle_cfg, product_cfg, check_tree_against_golden, rel_inf, logged_cut_group

pytestmark = pytest.mark.gpu

COEFF_TOL = 1e-10
QUERY_TOL = 1e-9


def points_in_cells(pts, cfg_kwargs, cells):
    """Mask of user-space points that fall into any of the (depth, centre) cells of the internal unit cube."""
    mn = np.asarray(cfg_kwargs.get("root_min", (-0.5,) * 3), np.float32).astype(np.float64)
    mx = np.asarray(cfg_kwargs.get("root_max", (0.5,) * 3), np.float32).astype(np.float64)
    u = (pts - (mn + mx) / 2) / (mx - mn)
    mask = np.zeros(len(pts), bool)
    for depth, c in cells:
        h = 0.5 ** (depth + 1)
        mask |= (np.abs(u - np.asarray(c)) <= h * (1 + 1e-9)).all(1)
    return mask


@pytest.fixture(scope="module")
def built(hp):
    """GPU-built trees, cached per case for the module."""
    cache = {}

    def get(name, **optkw):
        key = (name, tuple(sorted(optkw.items())))
        if key not in cache:
            cfg, prog = product_cfg(hp, name)
            t = hp.Octree()
            t.Create(cfg, prog, hp.BuildOpts(**optkw) if optkw else None)
            cache[key] = t
        return cache[key]
    return get


def test_sdf_program_evaluator_matches_cpu(hp, oracle):
    from oracle import hpref
    pts = np.random.default_rng(0).uniform(-0.6, 0.8, (20000, 3))
    for name in ("c1_readme", "c2_csg", "custom_domain"):
        items = CASES[name]["prog"]
        a = hp.SdfProgram(items).eval(pts)
        b = oracle.sdf_eval(hpref.make_program(items), pts)
        assert np.abs(a - b).max() <= 1e-14, name
    items = [("box", [0.1, 0.0, 0.0, 0.2, 0.3, 0.1]), ("sphere", [0.2, 0.1, 0, 0.25]), ("subtract", []),
             ("plane", [0.0, 0.0, 1.0, -0.05]), ("intersect", []), ("torus", [0, 0, 0, 0.3, 0.05, 2]), ("union", []), ("negate", [])]
    assert np.abs(hp.SdfProgram(items).eval(pts) - oracle.sdf_eval(hpref.make_program(items), pts)).max() <= 1e-14


def test_device_sqrt_is_the_correctly_rounded_ieee_square_root(hp):
    """sdf_eval.cuh: sdfSqrt replaces sqrt() in the SDF primitives (fast path of CUDA's sqrt without its range test and call
    scaffolding). |(x, 0, 0)| - 0 = sqrt(fl(x*x)) must equal numpy's correctly rounded sqrt bit for bit, over 300 decades."""
    rng = np.random.default_rng(123)
    n = 2_000_000
    x = np.concatenate([10.0 ** rng.uniform(-140, 140, n), rng.uniform(0, 2, n), [0.0, 1.0, 2.0, 4.0, 0.5, 1e-146, 1e150, 3.0, 1.0 + 2 ** -52]])
    pts = np.zeros((len(x), 3))
    pts[:, 0] = x
    got = hp.SdfProgram([("sphere", [0.0, 0.0, 0.0, 0.0])]).eval(pts)
    want = np.sqrt(x * x)
    bad = np.nonzero(got != want)[0]
    assert len(bad) == 0, (len(bad), x[bad[:5]], got[bad[:5]], want[bad[:5]])


def test_single_fits_match_reference_golden(hp):
    g = golden("fits")
    names = list(CASES)
    worst = 0.0
    for k in range(int(g["n_fits"])):
        case, degree, depth, degree_in = [int(v) for v in g["fit%03d_meta" % k]]
        if degree_in:
            continue        # kept-shell fits are exercised through Create (p-refinement) below
        cfg, prog = product_cfg(hp, names[case])
        coeffs, err, _ = hp.fit_batch(cfg, prog, g["fit%03d_cell" % k][None, :], [depth], degree)
        worst = max(worst, rel_inf(coeffs[0], g["fit%03d_coeffs" % k]))
        # the raw error is a sum of squares: where the SDF is exactly polynomial in the cell it is rounding noise
        floor = (1e-12 * np.abs(g["fit%03d_coeffs" % k]).max()) ** 2
        assert abs(err[0] - float(g["fit%03d_err" % k])) <= 1e-9 * float(g["fit%03d_err" % k]) + floor
    assert worst <= COEFF_TOL, worst


@pytest.mark.parametrize("degree", list(range(1, 12)))
def test_fit_batch_matches_oracle_all_degrees(hp, oracle, degree):
    """Every template instantiation of the fit kernel, incl. the 83-coefficient degree 6 and the multi-pass degrees. Seven
    fits at degrees 1..3 leave the last CTA partly filled (fitGroup packs 5, 3 and 3 fits per CTA there)."""
    from oracle import hpref
    cfg, prog = product_cfg(hp, "c2_csg")
    ocfg, oprog = oracle_cfg(hpref, "c2_csg")
    rng = np.random.default_rng(degree)
    depth = 5
    half = 0.5 ** (depth + 1)
    n = 7 if degree <= 3 else 6 if degree <= 6 else 2
    centres = (rng.integers(8, 24, (n, 3)) + 0.5) * 2 * half - 0.5
    cells = np.concatenate([centres, np.full((n, 1), half)], 1).astype(np.float32)
    coeffs, err, _ = hp.fit_batch(cfg, prog, cells, np.full(n, depth), degree)
    assert coeffs.shape[1] == hp.COEFF_COUNT[degree]
    for i in range(n):
        c, e = oracle.oracle_fit(ocfg, oprog, centres[i] - half, centres[i] + half, degree, depth)
        assert rel_inf(coeffs[i], c) <= COEFF_TOL
        assert abs(err[i] - e) <= 1e-9 * e + (1e-12 * np.abs(c).max()) ** 2


@pytest.mark.parametrize("name", ["sphere_poly_1e8", "custom_domain", "csg_small"])
def test_create_matches_reference_golden(hp, built, name):
    t = built(name)
    blk = hp.parse_block(t.ToMemoryBlockBytes())
    g = golden(name)
    worst, ndiv = check_tree_against_golden(blk, g, hp.COEFF_COUNT, COEFF_TOL, tree=t)
    st = t.stats()
    assert st["jobs_applied_p"] == int(g["applied_p"]) and st["jobs_applied_h"] == int(g["applied_h"])
    assert abs(st["total_error"] - float(g["final_total"])) <= 1e-6 * float(g["final_total"])
    q = t.Query(g["query_pts"])
    if ndiv == 0:
        assert np.abs(q - g["query_vals"]).max() <= QUERY_TOL
    else:   # points inside the (logged) divergent cells see another member of the tie group refined: exclude those cells
        bad = points_in_cells(g["query_pts"], CASES[name]["cfg"], logged_cut_group(t)[0])
        assert np.abs(q - g["query_vals"])[~bad].max() <= QUERY_TOL
    print(name, "worst |dc|inf/|c|inf", worst, "divergent cells (logged tie group at the cut):", ndiv, "rounds", st["rounds"], "fits", st["fits_evaluated"], "ms", st["total_ms"])


@pytest.mark.parametrize("name", ["sphere_exp_1e8", "c2_csg"])
def test_create_matches_oracle_full_tree(hp, oracle, built, name):
    """Whole-tree comparison against the CPU oracle run here: node arrays (numbering included), every leaf's
    coefficients, 1e5 query values; divergences would show in the decision log."""
    from oracle import hpref
    ocfg, oprog = oracle_cfg(hpref, name)
    o = oracle.OracleTree.build(ocfg, oprog, threads=8)
    t = built(name)
    a, b = hp.parse_block(t.ToMemoryBlockBytes()), hpref.parse_block(o.block())
    assert a["n_nodes"] == b["n_nodes"] and a["n_coeffs"] == b["n_coeffs"], (t.stats(), t.decision_log()[-3:])
    # canonical comparison (DFS by child slot): node NUMBERING may differ where two cells have errors equal to the last
    # bits (mirror-symmetric cells) and pop in the other order — same tree, children allocated in another order
    pa, da, ga, ca = leaf_table(a, hp.COEFF_COUNT)
    pb, db, gb, cb = leaf_table(b, hp.COEFF_COUNT)
    ma = {(path_code(p), int(d)): i for i, (p, d) in enumerate(zip(pa, da))}
    mb = {(path_code(p), int(d)): i for i, (p, d) in enumerate(zip(pb, db))}
    div = divergent_cells({k: int(ga[i]) for k, i in ma.items()}, {k: int(gb[i]) for k, i in mb.items()})
    allowed, _ = logged_cut_group(t)
    for code, d in div:      # identical topology, except inside the logged equal-error group at the termination cut
        assert cell_of(code, d) in allowed, ("unlogged divergence", cell_of(code, d), t.decision_log()[-6:])
    assert np.array_equal(np.bincount(ga, minlength=13), np.bincount(gb, minlength=13))
    worst = max(rel_inf(ca[i], cb[mb[k]]) for k, i in ma.items() if k in mb and k not in div)
    assert worst <= COEFF_TOL, worst
    same_numbering = all(np.array_equal(a["nodes"][f], b["nodes"][f]) for f in ("child", "deg", "depth"))
    la, lb = t.apply_log(), o.apply_log()
    assert la.shape == lb.shape
    # the same multiset of jobs was applied, with errors equal to rounding
    assert np.array_equal(np.sort(la[:, 1]), np.sort(lb[:, 1]))
    assert np.abs(np.sort(la[:, 4]) - np.sort(lb[:, 4])).max() <= 1e-9 * np.abs(lb[:, 4]).max()
    leaf = a["nodes"]["child"] == np.uint64(0xFFFFFFFFFFFFFFFF)
    pts = root_points(CASES[name]["cfg"], 100000, seed=5, margin=0.01)
    qa, qb = t.Query(pts), o.query(pts, 8)
    assert np.array_equal(qa == hp.DBL_MAX, qb == hp.DBL_MAX)
    ok = (qb != hp.DBL_MAX) & ~points_in_cells(pts, CASES[name]["cfg"], allowed if div else set())
    assert np.abs(qa - qb)[ok].max() <= QUERY_TOL
    so, st = o.stats(), t.stats()
    assert st["jobs_applied_p"] == so["applied_p"] and st["jobs_applied_h"] == so["applied_h"]
    assert st["n_leaves"] == int(leaf.sum())
    print(name, "worst", worst, "same node numbering:", same_numbering, "divergent cells:", len(div), "logged group:", len(allowed), {k: st[k] for k in ("rounds", "fits_evaluated", "jobs_evaluated", "total_ms", "fit_kernel_ms", "host_replay_ms", "near_tie_decisions", "cut_margin")})


@pytest.mark.parametrize("name", ["c1_readme", "csg_cont"])
def test_continuity_matches_reference_golden(hp, built, name):
    """PerformContinuityPostProcess: the converged solution of (M + lambda I) x = lambda c (CG to 1e-13) against the
    reference's, plus the gap of a reference-tolerance (1e-6) solve."""
    t = built(name, cg_tolerance=1e-13)
    g = golden(name)
    blk = hp.parse_block(t.ToMemoryBlockBytes())
    worst, ndiv = check_tree_against_golden(blk, g, hp.COEFF_COUNT, COEFF_TOL, tree=t)
    st = t.stats()
    assert st["cg_relative_residual"] <= 1e-13 and st["cg_iterations"] > 0
    if ndiv == 0:
        assert np.abs(t.Query(g["query_pts"]) - g["query_vals"]).max() <= QUERY_TOL
    t6 = built(name)                                                     # default tolerance = the reference's 1e-6f
    b6 = hp.parse_block(t6.ToMemoryBlockBytes())
    gap = np.abs(b6["coeffs"] - blk["coeffs"]).max()
    assert gap <= 1e-6 * np.abs(blk["coeffs"]).max() * 10
    # the reference starts CG from lambda * c (Octree.cpp:1755); the default here starts from c: same converged solution,
    # same stopping rule, fewer iterations
    tr = built(name, cg_tolerance=1e-13, cg_guess=hp.CG_GUESS_REFERENCE)
    br = hp.parse_block(tr.ToMemoryBlockBytes())
    assert np.abs(br["coeffs"] - blk["coeffs"]).max() <= 1e-12 * np.abs(blk["coeffs"]).max()
    t6r = built(name, cg_guess=hp.CG_GUESS_REFERENCE)
    assert t6.stats()["cg_iterations"] < t6r.stats()["cg_iterations"]
    print(name, "worst", worst, "cg its", st["cg_iterations"], "res", st["cg_relative_residual"], "ms", st["continuity_ms"],
          "tol-1e-6 gap", gap, "its", t6.stats()["cg_iterations"], "its with the reference's guess", t6r.stats()["cg_iterations"])


def test_build_option_switches_match_oracle(hp, oracle):
    from oracle import hpref
    ocfg, oprog = oracle_cfg(hpref, "sphere_poly_1e8")
    cfg, prog = product_cfg(hp, "sphere_poly_1e8")
    for kw in (dict(max_degree=3), dict(total_mode=1), dict(max_degree=2, max_depth=6)):
        o = oracle.OracleTree.build(ocfg, oprog, threads=8, **kw)
        t = hp.Octree()
        t.Create(cfg, prog, hp.BuildOpts(**kw))
        a, b = hp.parse_block(t.ToMemoryBlockBytes()), hpref.parse_block(o.block())
        assert a["n_nodes"] == b["n_nodes"] and a["n_coeffs"] == b["n_coeffs"], kw
        pa, da, ga, ca = leaf_table(a, hp.COEFF_COUNT)
        pb, db, gb, cb = leaf_table(b, hp.COEFF_COUNT)
        ma = {(path_code(p), int(d)): i for i, (p, d) in enumerate(zip(pa, da))}
        mb = {(path_code(p), int(d)): i for i, (p, d) in enumerate(zip(pb, db))}
        div = divergent_cells({k: int(ga[i]) for k, i in ma.items()}, {k: int(gb[i]) for k, i in mb.items()})
        allowed, _ = logged_cut_group(t)
        assert all(cell_of(c, d) in allowed for c, d in div), kw
        assert np.array_equal(np.bincount(ga, minlength=13), np.bincount(gb, minlength=13)), kw
        assert max(rel_inf(ca[i], cb[mb[k]]) for k, i in ma.items() if k in mb and k not in div) <= COEFF_TOL


@pytest.mark.parametrize("name", ["sphere_exp_1e8", "sphere_poly_1e8", "custom_domain"])
def test_mc_counter_nearness_matches_oracle(hp, oracle, name):
    """nearness_mode = HPSDF_NEARNESS_MC_COUNTER: the reference's 100-sample nearness estimator (Octree.cpp:1209-1247) on
    Philox points. The oracle side of this mode is bit-identical to the reference's own FApprox run on the same points
    (tests/test_oracle_vs_ref.py::test_mc_counter_nearness_bit_identical); the device evaluates the same estimator in the
    scheduler's ingest step. Same bar as the exact-mean mode: identical topology, coefficients 1e-10, Query 1e-9."""
    from oracle import hpref
    kw = CASES[name]["cfg"]
    if kw["nearness"] == 0:
        pytest.skip("nearness weighting is off in this case")
    ocfg, oprog = oracle_cfg(hpref, name)
    cfg, prog = product_cfg(hp, name)
    o = oracle.OracleTree.build(ocfg, oprog, threads=8, mc_seed=2017)
    t = hp.Octree()
    t.Create(cfg, prog, hp.BuildOpts(nearness_mode=hp.NEARNESS_MC_COUNTER, nearness_seed=2017))
    worst, ndiv = compare_with_oracle_tree(hp, t, o, kw)
    if name == "sphere_exp_1e8":
        # the same tree as the fixture generated by the reference's own sources (tests/golden/make_golden.py mc)
        g = golden("sphere_exp_1e8_mc2017")
        gw, gd = check_tree_against_golden(hp.parse_block(t.ToMemoryBlockBytes()), g, hp.COEFF_COUNT, COEFF_TOL, tree=t)
        assert gw <= COEFF_TOL
        if gd == 0:
            assert np.abs(t.Query(g["query_pts"]) - g["query_vals"]).max() <= QUERY_TOL
    exact = hp.Octree()
    exact.Create(cfg, prog)
    other = hp.Octree()
    other.Create(cfg, prog, hp.BuildOpts(nearness_mode=hp.NEARNESS_MC_COUNTER, nearness_seed=2018))
    sizes = [x.stats()["n_coeffs"] for x in (t, exact, other)]
    print(name, "nodes", t.stats()["n_nodes"], "coeffs (seed 2017, exact mean, seed 2018)", sizes, "worst", worst, "divergent (logged)", ndiv)
    # the host replay only sees fit records: the mode is refused there, loudly
    with pytest.raises(hp.HpsdfError) as e:
        hp.Octree().Create(cfg, prog, hp.BuildOpts(nearness_mode=hp.NEARNESS_MC_COUNTER, nearness_seed=1, scheduler=1))
    assert e.value.status == hp.ERR_UNSUPPORTED


@pytest.mark.parametrize("name", ["csg_small", "sphere_poly_1e8"])
def test_scheduling_knobs_do_not_change_the_tree(hp, built, name):
    """Round size (min_round_jobs), speculation and strict ordering only change WHEN a job is evaluated and node numbering:
    canonical topology and coefficients are those of the default schedule (outside the logged tie group at the cut)."""
    base = built(name)
    a = hp.parse_block(base.ToMemoryBlockBytes())
    pa, da, ga, ca = leaf_table(a, hp.COEFF_COUNT)
    ma = {(path_code(p), int(d)): i for i, (p, d) in enumerate(zip(pa, da))}
    for kw in (dict(min_round_jobs=1), dict(min_round_jobs=4096), dict(speculate=1), dict(strict_order=1, min_round_jobs=64), dict(jit=1, min_round_jobs=7)):
        t = built(name, **kw)
        b = hp.parse_block(t.ToMemoryBlockBytes())
        assert a["n_nodes"] == b["n_nodes"] and a["n_coeffs"] == b["n_coeffs"], kw
        pb, db, gb, cb = leaf_table(b, hp.COEFF_COUNT)
        mb = {(path_code(p), int(d)): i for i, (p, d) in enumerate(zip(pb, db))}
        div = divergent_cells({k: int(ga[i]) for k, i in ma.items()}, {k: int(gb[i]) for k, i in mb.items()})
        allowed = logged_cut_group(t)[0] | logged_cut_group(base)[0]
        assert all(cell_of(c, d) in allowed for c, d in div), kw
        assert max(rel_inf(ca[i], cb[mb[k]]) for k, i in ma.items() if k in mb and k not in div) <= 1e-12, kw
        assert t.stats()["jobs_applied_p"] == base.stats()["jobs_applied_p"] and t.stats()["jobs_applied_h"] == base.stats()["jobs_applied_h"], kw


def test_memory_block_is_accepted_by_the_cpu_side_and_back(hp, oracle, built):
    """ToMemoryBlock is byte-compatible: the oracle's (and, where built, the reference's own) FromMemoryBlock + Query
    accepts GPU-built trees; FromMemoryBlock accepts CPU-built trees."""
    from oracle import hpref
    t = built("csg_small")
    raw = t.ToMemoryBlockBytes()
    pts = root_points(CASES["csg_small"]["cfg"], 20000, seed=8, margin=0.02)
    qa = t.Query(pts)
    assert np.abs(oracle.OracleTree.from_block(raw).query(pts) - qa).max() <= QUERY_TOL
    if hpref.available():
        assert np.abs(hpref.RefTree.from_block(raw).query(pts) - qa).max() <= QUERY_TOL
    t2 = hp.Octree()
    t2.FromMemoryBlock(hp.MemoryBlock.frombytes(raw))
    assert np.array_equal(t2.Query(pts), qa)                          # round trip is bit-exact
    assert t2.ToMemoryBlockBytes()[:-80] == raw[:-80] or hp.parse_block(t2.ToMemoryBlockBytes())["n_coeffs"] == hp.parse_block(raw)["n_coeffs"]
    ocfg, oprog = oracle_cfg(hpref, "custom_domain")
    o = oracle.OracleTree.build(ocfg, oprog, threads=8)
    t3 = hp.Octree()
    t3.FromMemoryBlock(hp.MemoryBlock.frombytes(bytes(o.block())))
    p3 = root_points(CASES["custom_domain"]["cfg"], 20000, seed=9, margin=0.02)
    assert np.abs(t3.Query(p3) - o.query(p3)).max() <= QUERY_TOL
    mn, mx = t3.GetRootAABB()
    assert mn.tolist() == [-0.25] * 3 and mx.tolist() == [5.0] * 3
    c = t3.copy()                                                      # copy constructor (Octree.cpp:24-45)
    t3.Clear()
    assert np.abs(c.Query(p3) - o.query(p3)).max() <= QUERY_TOL


def test_bad_blocks_are_rejected(hp, built):
    raw = bytearray(built("csg_small").ToMemoryBlockBytes())
    for bad in (bytes(raw[:-8]), b"", bytes(raw[:50])):
        with pytest.raises(hp.HpsdfError) as e:
            hp.Octree().FromMemoryBlock(hp.MemoryBlock.frombytes(bad) if bad else hp.MemoryBlock(0, None))
        assert e.value.status == hp.ERR_BAD_BLOCK
    raw2 = bytearray(raw)
    n_coeffs = int(np.frombuffer(raw2[:8], np.uint64)[0])
    off = 16 + 8 * n_coeffs                                             # node 0
    raw2[off:off + 8] = np.uint64(10 ** 9).tobytes()                    # child index out of range
    with pytest.raises(hp.HpsdfError):
        hp.Octree().FromMemoryBlock(hp.MemoryBlock.frombytes(bytes(raw2)))
    for wrap in (2 ** 64 - 8, 2 ** 64 - 2):                             # child + 8 wraps around in u64: still rejected, not indexed
        raw3 = bytearray(raw)
        raw3[off:off + 8] = np.uint64(wrap).tobytes()
        with pytest.raises(hp.HpsdfError) as e:
            hp.Octree().FromMemoryBlock(hp.MemoryBlock.frombytes(bytes(raw3)))
        assert e.value.status == hp.ERR_BAD_BLOCK


def test_query_edge_cases(hp, oracle, built):
    from oracle import hpref
    t = built("sphere_poly_1e8")
    o = oracle.OracleTree.from_block(t.ToMemoryBlockBytes())
    assert len(t.Query(np.zeros((0, 3)))) == 0                         # empty batch
    edge = np.array([[0.5, 0.5, 0.5], [-0.5, -0.5, -0.5], [0.5000001, 0, 0], [0, 0, 0], [0.25, 0, 0], [-0.5, 0.5, 0.0],
                     [0.03125, 0.0625, -0.125], [1e-300, -1e-300, 0.0], [0.5 + 1e-9, 0, 0], [np.nextafter(0.5, 1), 0, 0],
                     [np.nan, 0, 0], [np.inf, 0, 0]])
    qa, qb = t.Query(edge), o.query(edge)
    assert np.array_equal(qa == hp.DBL_MAX, qb == hp.DBL_MAX)
    m = qb != hp.DBL_MAX
    assert np.abs(qa[m] - qb[m]).max() <= QUERY_TOL
    for n in (1, 255, 256, 257, 1000):                                  # ragged tiles
        pts = root_points(CASES["sphere_poly_1e8"]["cfg"], n, seed=n)
        assert np.abs(t.Query(pts) - o.query(pts)).max() <= QUERY_TOL
    assert isinstance(t.Query(np.array([0.1, 0.2, 0.3])), float)       # single point, like Octree::Query
    # every cell corner/face of the 16^3 grid and a finer lattice: descent ties (pt == midpoint) go to the upper child
    g = np.linspace(-0.5, 0.5, 65)
    lat = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    assert np.abs(t.Query(lat) - o.query(lat, 8)).max() <= QUERY_TOL


def test_query_gradient_matches_oracle(hp, oracle, built):
    t = built("csg_small")
    o = oracle.OracleTree.from_block(t.ToMemoryBlockBytes())
    pts = root_points(CASES["csg_small"]["cfg"], 5000, seed=4)
    va, ga = t.QueryWithGradient(pts)
    vb, gb = o.query_gradient(pts)
    assert np.abs(va - vb).max() <= QUERY_TOL
    assert np.abs(ga - gb).max() <= 1e-6                                # central differences amplify rounding by 1/(2 eps)


def test_large_batch_properties(hp, oracle, built):
    """BASELINE-scale batch (1.6e7 points): idempotent, chunk-independent, equal to the oracle on a subsample, and the
    device-pointer entry point gives the same bits as the host-pointer one."""
    import torch
    t = built("c2_csg")
    n = 1 << 24
    gen = torch.Generator(device="cuda").manual_seed(0x5DF0C7EE)
    pts = (torch.rand((n, 3), generator=gen, device="cuda", dtype=torch.float64) * 0.75 - 0.25).contiguous()
    out = torch.empty(n, device="cuda", dtype=torch.float64)
    t.QueryDevice(pts.data_ptr(), n, out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    out2 = torch.empty_like(out)
    t.QueryDevice(pts.data_ptr(), n, out2.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert torch.equal(out, out2)
    host = pts[: 1 << 22].cpu().numpy()
    assert np.array_equal(t.Query(host), out[: 1 << 22].cpu().numpy())
    o = oracle.OracleTree.from_block(t.ToMemoryBlockBytes())
    idx = np.random.default_rng(1).integers(0, n, 200000)
    sub = pts[torch.from_numpy(idx).cuda()].cpu().numpy()
    assert np.abs(o.query(sub, 8) - out[torch.from_numpy(idx).cuda()].cpu().numpy()).max() <= QUERY_TOL
    assert float(out.abs().max()) < 2.0                                 # all inside the root: no DBL_MAX
    # a point array that starts 8 bytes off a 16-byte boundary (a slice of a larger tensor) takes the scalar load path: same bits
    flat = torch.empty(3 * 100003 + 1, device="cuda", dtype=torch.float64)
    flat[1:] = pts[:100003].reshape(-1)
    odd = torch.empty(100003, device="cuda", dtype=torch.float64)
    assert (flat.data_ptr() + 8) % 16 == 8
    t.QueryDevice(flat.data_ptr() + 8, 100003, odd.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert torch.equal(odd, out[:100003])


def compare_with_oracle_tree(hp, t, o, cfg_kwargs, n_pts=100000, seed=5):
    """GPU tree `t` against oracle tree `o`: identical canonical topology (outside the logged tie group at the cut),
    per-leaf coefficients to COEFF_TOL, Query to QUERY_TOL. Returns (worst coefficient error, divergent cells)."""
    from oracle import hpref
    a, b = hp.parse_block(t.ToMemoryBlockBytes()), hpref.parse_block(o.block())
    assert a["n_nodes"] == b["n_nodes"] and a["n_coeffs"] == b["n_coeffs"], (a["n_nodes"], b["n_nodes"], a["n_coeffs"], b["n_coeffs"])
    pa, da, ga, ca = leaf_table(a, hp.COEFF_COUNT)
    pb, db, gb, cb = leaf_table(b, hp.COEFF_COUNT)
    ma = {(path_code(p), int(d)): i for i, (p, d) in enumerate(zip(pa, da))}
    mb = {(path_code(p), int(d)): i for i, (p, d) in enumerate(zip(pb, db))}
    div = divergent_cells({k: int(ga[i]) for k, i in ma.items()}, {k: int(gb[i]) for k, i in mb.items()})
    allowed, _ = logged_cut_group(t)
    for code, d in div:
        assert cell_of(code, d) in allowed, ("unlogged divergence", cell_of(code, d), t.decision_log()[-6:])
    assert np.array_equal(np.bincount(ga, minlength=13), np.bincount(gb, minlength=13))
    worst = max(rel_inf(ca[i], cb[mb[k]]) for k, i in ma.items() if k in mb and k not in div)
    assert worst <= COEFF_TOL, worst
    pts = root_points(cfg_kwargs, n_pts, seed=seed, margin=0.01)
    qa, qb = t.Query(pts), o.query(pts, 8)
    assert np.array_equal(qa == hp.DBL_MAX, qb == hp.DBL_MAX)
    ok = (qb != hp.DBL_MAX) & ~points_in_cells(pts, cfg_kwargs, allowed if div else set())
    assert np.abs(qa - qb)[ok].max() <= QUERY_TOL
    return worst, len(div)


@pytest.mark.parametrize("op", ["UnionSDF", "IntersectSDF", "SubtractSDF"])
def test_sdf_operations_match_oracle(hp, oracle, op):
    """Octree::UnionSDF / IntersectSDF / SubtractSDF (Octree.cpp:355-400) = re-Create from min / max of the old tree's
    Query and the new F. The configuration is the reference's own test (HPUnitTests.cpp:207-282: two radius-0.5 spheres at
    x = +-0.25, threshold 1e-8, nearness None, continuity off). The CPU oracle rebuilds from the SAME old tree (the
    GPU-built one, read through FromMemoryBlock) as its OCTREE primitive, so both sides approximate the same function:
    identical topology, coefficients to 1e-10, Query to 1e-9; the reference's 0.05 bound against the analytic min / max
    is kept as well."""
    from oracle import hpref
    kw = dict(threshold=1e-8, nearness=0, strength=0.0, continuity=False)
    cfg = hp.Config(target_error_threshold=1e-8, continuity_enforce=0)
    a = [("sphere", [0.25, 0.0, 0.0, 0.5])]
    b = [("sphere", [-0.25, 0.0, 0.0, 0.5])]
    t = hp.Octree()
    t.Create(cfg, hp.SdfProgram(a))
    old = oracle.OracleTree.from_block(t.ToMemoryBlockBytes())
    name = dict(UnionSDF="union", IntersectSDF="intersect", SubtractSDF="subtract")[op]
    o = oracle.OracleTree.build(hpref.make_config(threads=8, **kw), hpref.make_program(b + [("octree", [], old.h), (name, [])]), threads=8)
    getattr(t, op)(hp.SdfProgram(b))
    worst, ndiv = compare_with_oracle_tree(hp, t, o, kw)
    pts = np.random.default_rng(2).uniform(-0.5, 0.5, (100000, 3))
    fa = np.linalg.norm(pts - [0.25, 0, 0], axis=1) - 0.5
    fb = np.linalg.norm(pts + [0.25, 0, 0], axis=1) - 0.5
    truth = dict(UnionSDF=np.minimum(fa, fb), IntersectSDF=np.maximum(fa, fb), SubtractSDF=np.maximum(-fa, fb))[op]
    assert np.abs(t.Query(pts) - truth).max() <= 0.05
    print(op, "nodes", t.stats()["n_nodes"], "coeffs", t.stats()["n_coeffs"], "worst", worst, "divergent (logged)", ndiv)


def test_sdf_operation_keeps_build_options_and_survives_failure(hp):
    """The rebuild honours the caller's BuildOpts (max degree) and a failed rebuild leaves the tree as it was."""
    cfg = hp.Config(target_error_threshold=1e-6, continuity_enforce=0)
    t = hp.Octree()
    t.Create(cfg, hp.SdfProgram([("sphere", [0.25, 0.0, 0.0, 0.5])]), hp.BuildOpts(max_degree=3))
    t.UnionSDF(hp.SdfProgram([("sphere", [-0.25, 0.0, 0.0, 0.5])]), hp.BuildOpts(max_degree=3))
    blk = hp.parse_block(t.ToMemoryBlockBytes())
    leaf = blk["nodes"]["child"] == np.uint64(0xFFFFFFFFFFFFFFFF)
    assert blk["nodes"]["deg"][leaf].max() <= 3
    before = t.ToMemoryBlockBytes()
    with pytest.raises(hp.HpsdfError):
        t.UnionSDF(hp.SdfProgram([("torus", [0, 0, 0, 0.3, 0.1, 7])]))      # bad axis: the program does not resolve
    assert t.ToMemoryBlockBytes() == before


@pytest.mark.parametrize("name", ["sphere_poly_1e8", "custom_domain", "c2_csg"])
def test_query_ray_matches_oracle(hp, oracle, built, name):
    """Octree::QueryRay mirrored statement by statement (query_kernels.cuh: queryRayKernel): hit flags equal, t within the
    Query tolerance; a ray may differ only where a marched value sits within 1e-9 of a decision threshold (none expected)."""
    from oracle import hpref
    from test_oracle_vs_ref import ray_batch
    t = built(name)
    o = oracle.OracleTree.from_block(t.ToMemoryBlockBytes())
    org, d = ray_batch(CASES[name]["cfg"], 50000, 5)
    for t_max in (0.3, 10.0):
        hg, tg = t.QueryRay(org, d, t_max)
        ho, to = o.query_ray(org, d, t_max)
        differ = hg != ho
        assert differ.sum() <= 2, differ.sum()
        assert np.abs(tg - to)[~differ].max() <= QUERY_TOL
