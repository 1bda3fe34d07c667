"""GPU: every query of meshSampleKernel starts from its fit's cut of the 4-wide tree (meshCutKernel: up to 16 entries below
the root that can hold the closest triangle of some sample of the fit) with a pruning bound seeded from the distance at the
fit's centre. Neither may change which triangle wins, so fits with the cut must be bitwise equal to fits with
HPSDF_MESH_NO_CUT=1 (the walk from the root with no seed), in each phase of the kernel (see test_gpu_mesh_steps.py):

* "main": the tail phase off (HPSDF_MESH_NO_HANDOVER=1);
* "tail": the default, where handed-over stack entries can be cut records;
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


def set_mode(monkeypatch, mode, degree, cut):
    for k in ("HPSDF_MESH_NO_HANDOVER", "HPSDF_SAMPLE_CAP", "HPSDF_MESH_NO_CUT"):
        monkeypatch.delenv(k, raising=False)
    if mode == "main":
        monkeypatch.setenv("HPSDF_MESH_NO_HANDOVER", "1")
    elif mode == "small":
        monkeypatch.setenv("HPSDF_SAMPLE_CAP", str(3 * (4 * degree + 1) ** 3))
    if not cut:
        monkeypatch.setenv("HPSDF_MESH_NO_CUT", "1")


def assert_cut_changes_nothing(hp, monkeypatch, m, lo, hi, groups, mode, what, degrees=(2, 3, 4, 5, 6)):
    cfg = hp.Config(target_error_threshold=1e-6, continuity_enforce=0, root_min=tuple(lo), root_max=tuple(hi))
    prog = hp.SdfProgram([("mesh", [], m)])
    for degree in degrees:
        for cells, depth in groups:
            if degree >= 5 and len(cells) > 24:
                cells, depth = cells[::3], depth[::3]                 # keep the high degrees quick: every third depth-2 cell
            cells = cells.astype(np.float32)
            set_mode(monkeypatch, mode, degree, cut=True)
            c0, e0, _ = hp.fit_batch(cfg, prog, cells, depth, degree)
            set_mode(monkeypatch, mode, degree, cut=False)
            c1, e1, _ = hp.fit_batch(cfg, prog, cells, depth, degree)
            bad = np.flatnonzero(~(c0 == c1).all(1) | (e0 != e1))
            assert len(bad) == 0, "%s, %s: degree %d depth %d: %d of %d cells differ, first %s" % (
                what, mode, degree, depth[0], len(bad), len(cells), cells[bad[0]])


def grid_cells(depth):
    n = 2 ** depth
    idx = np.stack(np.meshgrid(*[np.arange(n)] * 3, indexing="ij"), -1).reshape(-1, 3)
    return np.concatenate([(idx + 0.5) / n - 0.5, np.full((len(idx), 1), 0.5 / n)], 1), np.full(len(idx), depth)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", list(MESHES) + ["dense_box"])
def test_cut_fits_equal_root_start_fits(hp, meshes, monkeypatch, name, mode):
    """The meshes of test_gpu_mesh_wide.py (the tetrahedron is the single-leaf root: its cut is that one leaf) and the dense
    box, on cells of depths 2, 4 and 6 in a root box twice the mesh."""
    v, m = meshes[name]
    lo, hi, groups = cells_for(v, np.random.default_rng(sum(map(ord, name))))
    assert_cut_changes_nothing(hp, monkeypatch, m, lo, hi, groups, mode, name)


@pytest.mark.parametrize("mode", MODES)
def test_far_cells_and_overflowing_cuts(hp, meshes, monkeypatch, mode):
    """A root box eight times the torus, so that most cells of depth 2 lie far outside the mesh and their bound U reaches
    across much of it; and the root cell and the depth-1 cells of the dense box, whose bound keeps every node of the top of
    the tree: the cut fills up and refuses expansions that would overflow it (it must stay a complete, shallower cut)."""
    v, m = meshes["torus"]
    lo, hi = (np.array(x) for x in mesh_root(v))
    c, e = (lo + hi) / 2, (hi - lo) / 2
    assert_cut_changes_nothing(hp, monkeypatch, m, c - 8 * e, c + 8 * e, [grid_cells(2)], mode, "far torus", degrees=(2, 4, 6))
    v, m = meshes["dense_box"]
    lo, hi = (np.array(x) for x in mesh_root(v))
    c, e = (lo + hi) / 2, (hi - lo) / 2
    groups = [(np.array([[0.0, 0.0, 0.0, 0.5]]), np.array([0])), grid_cells(1)]
    assert_cut_changes_nothing(hp, monkeypatch, m, c - 1.5 * e, c + 1.5 * e, groups, mode, "dense box, large cells")
