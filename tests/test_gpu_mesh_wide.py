"""GPU: the 4-wide mesh walk of meshSampleKernel against the per-thread binary walk of the generic sample kernel.

A program that is a single mesh is sampled by meshSampleKernel, the only reader of the 4-wide tree (128-byte nodes with
4-byte frame codes, mesh_build.cuh: meshWideKernel). The program [mesh, mesh, union] takes the generic sampleKernel, which
walks the binary tree per thread (mesh_eval.cuh: traverseThread), and union of a value with itself is that value. Both walks
return the closest triangle under (smallest f32 d², lowest triangle index) whatever their boxes, so the fitted coefficients
and errors must be bitwise equal: any box that cut off a closer triangle would show up here."""
import numpy as np
import pytest

from meshgen import bumpy_torus, mesh_root

pytestmark = pytest.mark.gpu


def box_mesh(k, half=0.3):
    """Closed axis-aligned cube, every face split into k x k squares of two triangles, counter-clockwise seen from outside:
    face normals ±x, ±y, ±z (the normal -z and the axis-aligned frames of the wide nodes)."""
    index, verts, tris = {}, [], []

    def vid(p):
        if p not in index:
            index[p] = len(verts)
            verts.append(p)
        return index[p]

    for a in range(3):
        b, c = (a + 1) % 3, (a + 2) % 3
        for side in (0, k):
            for i in range(k):
                for j in range(k):
                    q = []
                    for di, dj in ((0, 0), (1, 0), (1, 1), (0, 1)):
                        p = [0, 0, 0]
                        p[a], p[b], p[c] = side, i + di, j + dj
                        q.append(vid(tuple(p)))
                    if side == k:           # b x c = +a: counter-clockwise in (b, c) faces +a
                        tris += [(q[0], q[1], q[2]), (q[0], q[2], q[3])]
                    else:
                        tris += [(q[0], q[2], q[1]), (q[0], q[3], q[2])]
    v = (np.array(verts, np.float64) / k * 2 - 1) * half
    return v.astype(np.float32), np.array(tris, np.uint32)


def tetrahedron(s=0.3):
    """Closed mesh of 4 triangles: one BVH leaf, so the wide tree is the single-leaf root."""
    v = np.array([[1, 1, 1], [1, -1, -1], [-1, 1, -1], [-1, -1, 1]], np.float64) * s
    tris = []
    for f in ((0, 1, 2), (0, 1, 3), (0, 2, 3), (1, 2, 3)):
        other = ({0, 1, 2, 3} - set(f)).pop()
        a, b, c = v[list(f)]
        if np.dot(np.cross(b - a, c - a), a - v[other]) < 0:
            f = (f[0], f[2], f[1])
        tris.append(f)
    return v.astype(np.float32), np.array(tris, np.uint32)


MESHES = {
    "torus": lambda: bumpy_torus(60, 40),
    "fine_torus": lambda: bumpy_torus(400, 174),
    "box": lambda: box_mesh(24),
    "tetrahedron": tetrahedron,
}


@pytest.fixture(scope="module")
def meshes(hp):
    out = {}
    for name, make in MESHES.items():
        v, t = make()
        out[name] = (v, hp.Mesh(v, t))
    return out


def cells_for(v, rng):
    """Cells of the root box around the mesh (mesh_root, widened 2x so that part of it is far field): every cell of depth 2
    (far field, and cells straddling the surface), and random cells of depths 4 and 6 centred near the surface or anywhere."""
    lo, hi = (np.array(x) for x in mesh_root(v))
    c, e = (lo + hi) / 2, (hi - lo) / 2
    lo, hi = c - 2 * e, c + 2 * e
    groups = []
    for depth, count in ((2, None), (4, 24), (6, 24)):
        half = 0.5 ** (depth + 1)
        n = 2 ** depth
        if count is None:
            idx = np.stack(np.meshgrid(*[np.arange(n)] * 3, indexing="ij"), -1).reshape(-1, 3)
        else:
            near = (v[rng.integers(0, len(v), count // 2)] - lo) / (hi - lo)                  # unit-cube coordinates of vertices
            idx = np.concatenate([np.clip((near * n).astype(int), 0, n - 1), rng.integers(0, n, (count - count // 2, 3))])
        centres = (idx + 0.5) * 2 * half - 0.5
        groups.append((np.concatenate([centres, np.full((len(idx), 1), half)], 1), np.full(len(idx), depth)))
    return lo, hi, groups


@pytest.mark.parametrize("name", list(MESHES))
def test_wide_walk_fits_equal_binary_walk_fits(hp, meshes, name):
    v, m = meshes[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    lo, hi, groups = cells_for(v, rng)
    cfg = hp.Config(target_error_threshold=1e-6, continuity_enforce=0, root_min=tuple(lo), root_max=tuple(hi))
    wide = hp.SdfProgram([("mesh", [], m)])
    binary = hp.SdfProgram([("mesh", [], m), ("mesh", [], m), ("union", [])])
    for degree in (2, 3, 4, 5, 6):
        for cells, depth in groups:
            if degree >= 5 and len(cells) > 24:
                cells, depth = cells[::3], depth[::3]                 # keep the high degrees quick: every third depth-2 cell
            cells = cells.astype(np.float32)
            c0, e0, _ = hp.fit_batch(cfg, wide, cells, depth, degree)
            c1, e1, _ = hp.fit_batch(cfg, binary, cells, depth, degree)
            bad = np.flatnonzero(~(c0 == c1).all(1) | (e0 != e1))
            assert len(bad) == 0, "%s degree %d depth %d: %d of %d cells differ, first %s" % (name, degree, depth[0], len(bad), len(cells), cells[bad[0]])
