"""GPU: parity at the sizes bench.py measures (BASELINE.json configs[2..4] on their procedural stand-ins, SURVEY.md §8d).

* C3 (870 000 triangles, threshold 1e-6, continuity strength 8): the whole tree against the CPU oracle (tens of seconds of
  host time on the box's cores).
* C4 (1.6 M triangles, threshold 1e-8, max degree 6): far too large for a CPU build inside a test, so parity is sampled:
  200 random leaves of the GPU tree are refitted with the CPU oracle's FitPolynomial over its Mesh + BVH (the restatement
  that tests/test_oracle_golden.py pins to the reference's own output), replaying each leaf's history from the build's apply
  log (from-scratch fit, then kept-shell fits), and the oracle's FromMemoryBlock + Query reads the GPU tree back.
* C5: the Philox point stream is the numpy statement's, chunking / sharding do not change a single value.
"""
import os

import numpy as np
import pytest

from cases import leaf_table, path_code, divergent_cells, cell_of
from common import rel_inf, logged_cut_group
from meshgen import bumpy_torus, mesh_root
import philox

pytestmark = pytest.mark.gpu

NOCHILD = np.uint64(0xFFFFFFFFFFFFFFFF)
THREADS = os.cpu_count() or 1


def test_c3_full_size_tree_matches_the_oracle(hp, oracle):
    from oracle import hpref
    v, t = bumpy_torus(1000, 435)
    lo, hi = mesh_root(v)
    m = hp.Mesh(v, t)
    om = oracle.OracleMesh(v, t)
    kw = dict(threshold=1e-6, nearness=0, strength=0.0, continuity=True, cstrength=8.0, root_min=lo, root_max=hi)
    o = oracle.OracleTree.build(hpref.make_config(threads=THREADS, **kw), hpref.make_program([("mesh", [], om.h)]), threads=THREADS, cg_tol=1e-14)
    cfg = hp.Config(target_error_threshold=1e-6, continuity_enforce=1, continuity_strength=8.0, root_min=lo, root_max=hi)
    tree = hp.Octree()
    # (the per-leaf relative measure below amplifies the solvers' residuals on leaves with small coefficients: two solves to a
    # relative residual of 1e-13 that start from different guesses differ by 1.1e-10 there; while the GPU started from the
    # checker's own guess the two iterate sequences — and their errors — were nearly the same. Both sides go one decade further.)
    tree.Create(cfg, hp.SdfProgram([("mesh", [], m)]), hp.BuildOpts(cg_tolerance=1e-14))
    assert tree.stats()["cg_relative_residual"] <= 1e-14
    a, b = hp.parse_block(tree.ToMemoryBlockBytes()), hpref.parse_block(o.block())
    assert a["n_nodes"] == b["n_nodes"] and a["n_coeffs"] == b["n_coeffs"]
    pa, da, ga, ca = leaf_table(a, hp.COEFF_COUNT)
    pb, db, gb, cb = leaf_table(b, hp.COEFF_COUNT)
    ma = {(path_code(p), int(d)): i for i, (p, d) in enumerate(zip(pa, da))}
    mb = {(path_code(p), int(d)): i for i, (p, d) in enumerate(zip(pb, db))}
    div = divergent_cells({k: int(ga[i]) for k, i in ma.items()}, {k: int(gb[i]) for k, i in mb.items()})
    allowed, _ = logged_cut_group(tree)
    for code, d in div:
        assert cell_of(code, d) in allowed, ("unlogged divergence", cell_of(code, d))
    worst = max(rel_inf(ca[i], cb[mb[k]]) for k, i in ma.items() if k in mb and k not in div)
    assert worst <= 1e-10, worst
    pts = np.random.default_rng(3).uniform(lo, hi, (200000, 3))
    dq = np.abs(tree.Query(pts) - o.query(pts, THREADS))
    if div:
        from test_gpu_parity import points_in_cells
        dq = dq[~points_in_cells(pts, kw, allowed)]
    assert dq.max() <= 1e-9
    print("C3 full size: nodes", a["n_nodes"], "coeffs", a["n_coeffs"], "divergent (logged)", len(div), "worst |dc|/|c|", worst, "max |dQuery|", dq.max(),
          "cg iterations", tree.stats()["cg_iterations"], "residual", tree.stats()["cg_relative_residual"])


def leaf_histories(blk, log):
    """Per leaf node index: (d0, d1) = degree of the from-scratch fit that created its coefficients and its final degree.
    Coarse cells start at degree 2 (Octree.cpp:840); children of an H job start at the parent's degree (:820); every P job
    on the node adds one kept-shell fit (:846-851)."""
    nodes = blk["nodes"]
    d0 = {}
    for row in log:
        idx, kind, deg = int(row[0]), int(row[1]), int(row[2])
        if kind == 1:
            c = int(nodes["child"][idx])
            for k in range(8):
                d0[c + k] = deg
    out = {}
    for i in np.nonzero(nodes["child"] == NOCHILD)[0]:
        out[int(i)] = (d0.get(int(i), 2), int(nodes["deg"][i]))
    return out


def refit_chain(oracle, cfg, prog, mn, mx, d0, d1, depth):
    """One leaf's history replayed with the oracle's FitPolynomial: from scratch at degree d0, then kept-shell fits up to d1."""
    coeffs, kept = None, 0
    for d in range(d0, d1 + 1):
        coeffs, _ = oracle.oracle_fit(cfg, prog, mn, mx, d, depth, kept, coeffs)
        kept = d
    return coeffs


def test_c4_full_size_sampled_refit_with_the_oracle(hp, oracle):
    from concurrent.futures import ThreadPoolExecutor
    from oracle import hpref
    v, t = bumpy_torus(1000, 800)
    lo, hi = mesh_root(v)
    m = hp.Mesh(v, t)
    cfg = hp.Config(target_error_threshold=1e-8, continuity_enforce=0, root_min=lo, root_max=hi)
    tree = hp.Octree()
    tree.Create(cfg, hp.SdfProgram([("mesh", [], m)]), hp.BuildOpts(max_degree=6))
    raw = tree.ToMemoryBlockBytes()
    blk = hp.parse_block(raw)
    hist = leaf_histories(blk, tree.apply_log())
    leaves = np.array(sorted(hist))
    assert blk["nodes"]["deg"][leaves].max() <= 6
    pick = np.random.default_rng(11).choice(leaves, 200, replace=False)
    om = oracle.OracleMesh(v, t)
    ocfg = hpref.make_config(threshold=1e-8, continuity=False, root_min=lo, root_max=hi, threads=THREADS)
    oprog = hpref.make_program([("mesh", [], om.h)])
    nodes = blk["nodes"]
    oracle.tables()                   # initialises the oracle's constant tables before the threads below share them
    with ThreadPoolExecutor(THREADS) as pool:       # ctypes releases the GIL: the fits run in parallel
        coeffs = list(pool.map(lambda i: refit_chain(oracle, ocfg, oprog, nodes["mn"][i], nodes["mx"][i], hist[int(i)][0], hist[int(i)][1],
                                                     int(nodes["depth"][i])), pick))
    worst = 0.0
    for k, i in enumerate(pick):
        s, n = int(nodes["cstart"][i]), hp.COEFF_COUNT[int(nodes["deg"][i])]
        worst = max(worst, rel_inf(blk["coeffs"][s:s + n], coeffs[k]))
    assert worst <= 1e-10, worst
    # the oracle's FromMemoryBlock + Query on the GPU-built tree
    ot = oracle.OracleTree.from_block(raw)
    pts = np.random.default_rng(12).uniform(lo, hi, (200000, 3))
    dq = np.abs(ot.query(pts, THREADS) - tree.Query(pts)).max()
    assert dq <= 1e-9, dq
    st = tree.stats()
    print("C4 full size: nodes", st["n_nodes"], "coeffs", st["n_coeffs"], "ms", st["total_ms"], "| 200 leaves refitted by the oracle: worst |dc|/|c|",
          worst, "| oracle Query of the GPU tree: max |d|", dq, "| degrees of the sample", np.bincount(nodes["deg"][pick], minlength=7).tolist())


def test_philox_points_are_the_numpy_stream_and_sharding_invariant(hp):
    import torch
    lo, hi = (-0.41, -0.4, -0.72), (0.43, 0.5, 0.7)
    n = 1 << 20
    seed = 0x5DF0C7EE
    buf = torch.empty((n, 3), device="cuda", dtype=torch.float64)
    s = torch.cuda.current_stream().cuda_stream
    hp.uniform_points_device(seed, 0, n, lo, hi, buf.data_ptr(), s)
    torch.cuda.synchronize()
    got = buf.cpu().numpy()
    assert np.array_equal(got[:50000], philox.uniform_points(seed, 0, 50000, lo, hi))
    assert np.array_equal(got[-1000:], philox.uniform_points(seed, n - 1000, 1000, lo, hi))
    # a shard that starts beyond 2^32 uses the high counter word
    big = (1 << 32) + 12345
    hp.uniform_points_device(seed, big, 4096, lo, hi, buf.data_ptr(), s)
    torch.cuda.synchronize()
    assert np.array_equal(buf[:4096].cpu().numpy(), philox.uniform_points(seed, big, 4096, lo, hi))
    # sharded generation (3 ranks' contiguous ranges) = the single stream
    parts = []
    for r in range(3):
        b, e = hp.shard_range(n, r, 3)
        hp.uniform_points_device(seed, b, e - b, lo, hi, buf.data_ptr(), s)
        torch.cuda.synchronize()
        parts.append(buf[: e - b].cpu().numpy().copy())
    assert np.array_equal(np.concatenate(parts), got)
    assert (got >= np.array(lo)).all() and (got < np.array(hi)).all()
