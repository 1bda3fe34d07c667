"""GPU: the node step of meshSampleKernel puts leaf children straight into its 8-entry leaf queue, and a stale stack entry
is dropped together with the farther siblings pushed by the same node step. Neither may change which triangle wins, so
fits through the 4-wide walk must stay bitwise equal to fits through the per-thread binary walk ([mesh, mesh, union],
see test_gpu_mesh_wide.py), with each phase of the kernel checked on its own:

* "main": the tail phase off (HPSDF_MESH_NO_HANDOVER=1), every query walked by its own lane;
* "tail": the default, where lanes that ran out of samples take stack entries (sub-trees) from lanes that still have some;
* "small": launches of three fits (HPSDF_SAMPLE_CAP), so that the tail phase does most of the work."""
import numpy as np
import pytest

from meshgen import mesh_root
from test_gpu_mesh_wide import MESHES, box_mesh, cells_for

pytestmark = pytest.mark.gpu

MODES = ("main", "tail", "small")


@pytest.fixture(scope="module")
def meshes(hp):
    out = {}
    for name, make in list(MESHES.items()) + [("dense_box", lambda: box_mesh(64))]:
        v, t = make()
        out[name] = (v, hp.Mesh(v, t))
    return out


def set_mode(monkeypatch, mode, degree):
    monkeypatch.delenv("HPSDF_MESH_NO_HANDOVER", raising=False)
    monkeypatch.delenv("HPSDF_SAMPLE_CAP", raising=False)
    if mode == "main":
        monkeypatch.setenv("HPSDF_MESH_NO_HANDOVER", "1")
    elif mode == "small":
        monkeypatch.setenv("HPSDF_SAMPLE_CAP", str(3 * (4 * degree + 1) ** 3))


def assert_walks_agree(hp, monkeypatch, m, lo, hi, groups, mode, what):
    cfg = hp.Config(target_error_threshold=1e-6, continuity_enforce=0, root_min=tuple(lo), root_max=tuple(hi))
    wide = hp.SdfProgram([("mesh", [], m)])
    binary = hp.SdfProgram([("mesh", [], m), ("mesh", [], m), ("union", [])])
    for degree in (2, 3, 4, 5, 6):
        for cells, depth in groups:
            if degree >= 5 and len(cells) > 24:
                cells, depth = cells[::3], depth[::3]                 # keep the high degrees quick: every third depth-2 cell
            cells = cells.astype(np.float32)
            set_mode(monkeypatch, mode, degree)
            c0, e0, _ = hp.fit_batch(cfg, wide, cells, depth, degree)
            monkeypatch.delenv("HPSDF_SAMPLE_CAP", raising=False)
            c1, e1, _ = hp.fit_batch(cfg, binary, cells, depth, degree)
            bad = np.flatnonzero(~(c0 == c1).all(1) | (e0 != e1))
            assert len(bad) == 0, "%s, %s: degree %d depth %d: %d of %d cells differ, first %s" % (
                what, mode, degree, depth[0], len(bad), len(cells), cells[bad[0]])


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", list(MESHES))
def test_wide_walk_fits_equal_binary_walk_fits_per_phase(hp, meshes, monkeypatch, name, mode):
    v, m = meshes[name]
    lo, hi, groups = cells_for(v, np.random.default_rng(sum(map(ord, name))))
    assert_walks_agree(hp, monkeypatch, m, lo, hi, groups, mode, name)


@pytest.mark.parametrize("mode", MODES)
def test_full_leaf_queues_on_a_dense_box(hp, meshes, monkeypatch, mode):
    """A closed cube of 49 152 triangles. The root cell and the cells of depth 2 hold samples inside the cube and on its planes
    of symmetry, where many leaves lie at the same distance: lanes meet bottom-level nodes full of leaves that pass the bound,
    fill their leaf queues and wait for triangle iterations, and ties (lowest triangle index wins) are common."""
    v, m = meshes["dense_box"]
    lo, hi = (np.array(x) for x in mesh_root(v))
    c, e = (lo + hi) / 2, (hi - lo) / 2
    lo, hi = c - 2 * e, c + 2 * e
    n = 4
    idx = np.stack(np.meshgrid(*[np.arange(n)] * 3, indexing="ij"), -1).reshape(-1, 3)
    depth2 = np.concatenate([(idx + 0.5) / n - 0.5, np.full((len(idx), 1), 0.5 / n)], 1)
    groups = [(np.array([[0.0, 0.0, 0.0, 0.5]]), np.array([0])), (depth2, np.full(len(idx), 2))]
    assert_walks_agree(hp, monkeypatch, m, lo, hi, groups, mode, "dense box")
