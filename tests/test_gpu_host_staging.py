"""The host-array entry points (Query, QueryWithGradient, QueryDerivatives, QueryRay, Raycast, SdfProgram.eval,
Mesh.SignedDistanceAtPt) cut a large call into chunks of at least 2^16 items over three streams. A call of 6 * 2^16 + 123
items runs as seven chunks: the streams rotate more than twice and the last chunk is ragged. Its result must equal,
bit for bit, the concatenation of one-chunk calls on slices of 2^16 items."""
import ctypes as C

import numpy as np
import pytest

from cases import CASES, root_points
from common import product_cfg
from meshgen import bumpy_torus, mesh_root

pytestmark = pytest.mark.gpu

N = 6 * 2 ** 16 + 123
SLICE = 2 ** 16


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))


@pytest.fixture(scope="module")
def setup(hp):
    cfg, prog = product_cfg(hp, "csg_small")
    tree = hp.Octree()
    tree.Create(cfg, prog)
    v, t = bumpy_torus(60, 40)
    mesh = hp.Mesh(v, t)
    k = CASES["csg_small"]["cfg"]
    pts = root_points(k, N, seed=5, margin=0.1)                 # about a third of them outside the root
    rng = np.random.default_rng(6)
    dirs = rng.normal(size=(N, 3))
    mlo, mhi = mesh_root(v)
    mpts = rng.uniform(np.array(mlo) - 0.1, np.array(mhi) + 0.1, (N, 3)).astype(np.float32)
    return hp, tree, prog, mesh, pts, dirs, mpts


def raycast(hp, tree, o, d, normals):
    """hpsdf_raycast with or without the optional normals."""
    t = np.empty(len(o), np.float64)
    nrm = np.empty((len(o), 3), np.float64) if normals else None
    hp._check(hp.lib().hpsdf_raycast(tree._h, o.ctypes.data, d.ctypes.data, len(o), 0.0, np.inf, 0.0, t.ctypes.data,
                                     nrm.ctypes.data if normals else None))
    return (t, nrm) if normals else (t,)


def entry_points(hp, tree, prog, mesh, pts, dirs, mpts):
    """name -> function of a slice [a, b) returning the outputs of one call on it."""
    origins = pts * 1.5
    return {
        "Query": lambda a, b: (tree.Query(pts[a:b]),),
        "QueryWithGradient": lambda a, b: tree.QueryWithGradient(pts[a:b]),
        "QueryDerivatives": lambda a, b: tree.QueryDerivatives(pts[a:b]),
        "QueryDerivatives(hessian)": lambda a, b: tree.QueryDerivatives(pts[a:b], hessian=True),
        "QueryRay": lambda a, b: tree.QueryRay(origins[a:b], dirs[a:b], 2.0),
        "Raycast": lambda a, b: raycast(hp, tree, np.ascontiguousarray(origins[a:b]), np.ascontiguousarray(dirs[a:b]), False),
        "Raycast(normals)": lambda a, b: raycast(hp, tree, np.ascontiguousarray(origins[a:b]), np.ascontiguousarray(dirs[a:b]), True),
        "SdfProgram.eval": lambda a, b: (prog.eval(pts[a:b]),),
        "Mesh.SignedDistanceAtPt": lambda a, b: (mesh.SignedDistanceAtPt(mpts[a:b]),),
    }


def test_chunked_calls_equal_one_chunk_calls(setup):
    hp, tree, prog, mesh, pts, dirs, mpts = setup
    calls = entry_points(hp, tree, prog, mesh, pts, dirs, mpts)
    # interleaved on one device: each call reuses staging that a call with another item size used before it
    whole = {name: f(0, N) for name, f in calls.items()}
    parts = {name: [] for name in calls}
    for a in range(0, N, SLICE):
        for name, f in calls.items():
            parts[name].append(f(a, min(a + SLICE, N)))
    for name in calls:
        for k, got in enumerate(whole[name]):
            want = np.concatenate([p[k] for p in parts[name]])
            assert same_bits(got, want), (name, k)
    outside = (tree.Query(pts) == hp.DBL_MAX)
    assert 0.2 < outside.mean() < 0.6


def test_gradients_outside_the_root_are_zero_after_a_call_inside(setup):
    hp, tree, prog, mesh, pts, dirs, mpts = setup
    inside = root_points(CASES["csg_small"]["cfg"], N, seed=8, margin=-0.05)
    v, g = tree.QueryWithGradient(inside)
    assert (v != hp.DBL_MAX).all() and (np.abs(g).sum(1) > 0).mean() > 0.9
    outside = inside + 2.0
    v, g = tree.QueryWithGradient(outside)
    assert (v == hp.DBL_MAX).all()
    assert (g == 0.0).all()


def test_empty_calls(setup):
    hp, tree, prog, mesh, pts, dirs, mpts = setup
    L = hp.lib()
    x, d = pts[:2].copy(), dirs[:2].copy()
    v, g, h, hit = np.empty(2), np.empty((2, 3)), np.empty((2, 6)), np.empty(2, np.uint8)
    mx, mo = mpts[:2].copy(), np.empty(2, np.float32)
    valid = {
        "hpsdf_query": lambda: L.hpsdf_query(tree._h, x.ctypes.data, 0, v.ctypes.data),
        "hpsdf_query_with_gradient": lambda: L.hpsdf_query_with_gradient(tree._h, x.ctypes.data, 0, v.ctypes.data, g.ctypes.data),
        "hpsdf_query_derivatives": lambda: L.hpsdf_query_derivatives(tree._h, x.ctypes.data, 0, v.ctypes.data, g.ctypes.data, h.ctypes.data),
        "hpsdf_query_ray": lambda: L.hpsdf_query_ray(tree._h, x.ctypes.data, d.ctypes.data, 0, 1.0, hit.ctypes.data, v.ctypes.data),
        "hpsdf_raycast": lambda: L.hpsdf_raycast(tree._h, x.ctypes.data, d.ctypes.data, 0, 0.0, 1.0, 0.0, v.ctypes.data, g.ctypes.data),
        "hpsdf_sdf_eval": lambda: L.hpsdf_sdf_eval(C.byref(prog._c), x.ctypes.data, 0, v.ctypes.data, -1),
        "hpsdf_mesh_signed_distance": lambda: L.hpsdf_mesh_signed_distance(mesh._h, mx.ctypes.data, 0, mo.ctypes.data),
    }
    for name, call in valid.items():
        assert call() == hp.OK, name
    # null arrays at n = 0: hpsdf_sdf_eval rejects them, the others accept them
    null = {
        "hpsdf_query": (lambda: L.hpsdf_query(tree._h, None, 0, None), hp.OK),
        "hpsdf_query_with_gradient": (lambda: L.hpsdf_query_with_gradient(tree._h, None, 0, None, None), hp.OK),
        "hpsdf_query_derivatives": (lambda: L.hpsdf_query_derivatives(tree._h, None, 0, None, None, None), hp.OK),
        "hpsdf_query_ray": (lambda: L.hpsdf_query_ray(tree._h, None, None, 0, 1.0, None, None), hp.OK),
        "hpsdf_raycast": (lambda: L.hpsdf_raycast(tree._h, None, None, 0, 0.0, 1.0, 0.0, None, None), hp.OK),
        "hpsdf_sdf_eval": (lambda: L.hpsdf_sdf_eval(C.byref(prog._c), None, 0, None, -1), hp.ERR_INVALID_ARG),
        "hpsdf_mesh_signed_distance": (lambda: L.hpsdf_mesh_signed_distance(mesh._h, None, 0, None), hp.OK),
    }
    for name, (call, want) in null.items():
        assert call() == want, name
