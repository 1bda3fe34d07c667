"""GPU: the host replay (scheduler = 1) against the device-resident scheduler on a mesh program. Both launch their rounds'
fits through the same code, whose degree groups of a mesh round run concurrently on their own slices of the sample scratch
(or, with HPSDF_SAMPLE_CAP set, one after another in chunks). Fits are independent and both schedulers fit the same cells
with the same kernels, so the trees must agree bit for bit outside the logged equal-error group at the termination cut."""
import numpy as np
import pytest

from cases import leaf_table, path_code, cell_of, divergent_cells
from common import logged_cut_group
from meshgen import bumpy_torus, mesh_root

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torus(hp):
    v, t = bumpy_torus(60, 40)
    return v, hp.Mesh(v, t)


@pytest.mark.parametrize("sample_cap", [None, 50000])
def test_host_replay_builds_the_device_schedulers_mesh_tree(hp, torus, monkeypatch, sample_cap):
    v, m = torus
    lo, hi = mesh_root(v)
    if sample_cap is None:
        monkeypatch.delenv("HPSDF_SAMPLE_CAP", raising=False)
    else:
        monkeypatch.setenv("HPSDF_SAMPLE_CAP", str(sample_cap))
    cfg = hp.Config(target_error_threshold=1e-8, nearness_type=0, continuity_enforce=0, root_min=lo, root_max=hi)
    prog = hp.SdfProgram([("mesh", [], m)])
    trees = {}
    for sched in (0, 1):
        trees[sched] = hp.Octree()
        trees[sched].Create(cfg, prog, hp.BuildOpts(scheduler=sched, min_round_jobs=64))
    dev, host = trees[0], trees[1]
    # several rounds after the coarse one; 4096 coarse jobs of one fit each, and some later job with 8 child fits at its
    # degree and a p-fit at the next one, so that its round had at least two degree groups
    hs = host.stats()
    assert hs["rounds"] >= 3, hs
    assert hs["fits_evaluated"] - 4096 > 8 * (hs["jobs_evaluated"] - 4096), hs
    a, b = hp.parse_block(dev.ToMemoryBlockBytes()), hp.parse_block(host.ToMemoryBlockBytes())
    assert a["n_nodes"] == b["n_nodes"] and a["n_coeffs"] == b["n_coeffs"]
    pa, da, ga, ca = leaf_table(a, hp.COEFF_COUNT)
    pb, db, gb, cb = leaf_table(b, hp.COEFF_COUNT)
    ma = {(path_code(p), int(d)): i for i, (p, d) in enumerate(zip(pa, da))}
    mb = {(path_code(p), int(d)): i for i, (p, d) in enumerate(zip(pb, db))}
    div = divergent_cells({k: int(ga[i]) for k, i in ma.items()}, {k: int(gb[i]) for k, i in mb.items()})
    allowed = logged_cut_group(dev)[0] | logged_cut_group(host)[0]
    assert all(cell_of(c, d) in allowed for c, d in div), div
    same = [k for k in ma if k in mb and k not in div]
    assert len(same) > 0.9 * len(ma)
    assert all(np.array_equal(ca[ma[k]], cb[mb[k]]) for k in same)
    assert dev.stats()["jobs_applied_p"] == host.stats()["jobs_applied_p"] and dev.stats()["jobs_applied_h"] == host.stats()["jobs_applied_h"]
