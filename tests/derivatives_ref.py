"""Numpy checker of the hpsdf_query_derivatives contract (DESIGN §13). It shares no code with the kernel: the leaf is found
in the MemoryBlock with the reference's descent (Octree.cpp:662-702: f32 containment test, then the f64 coordinate against
the f32 cell midpoint), and P, grad P and the Hessian of P come from numpy.polynomial.legendre (legval / legder) with the
NormalisedLengths scale sqrt((2j+1) 2^depth) and the BasisIndexValues order. Every component also comes with the sum of
the absolute values of its terms, which sets the tolerance of a comparison."""
import numpy as np
from numpy.polynomial import legendre as L

INTERNAL = 13
COUNTS = [1, 4, 10, 20, 35, 56, 83, 120, 165, 220, 286, 364, 455]
HESS_AXES = [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]      # xx, xy, xz, yy, yz, zz
DBL_MAX = np.finfo(np.float64).max


def basis_index(degree):
    """(a, b, c) Legendre degrees of x, y, z per coefficient: shell by shell, a then b, c = p - a - b; 83 at degree 6."""
    out = [(a, b, p - a - b) for p in range(degree + 1) for a in range(p + 1) for b in range(p - a + 1)]
    return np.array(out[:COUNTS[degree]], np.int64)


def root_map(root_min, root_max):
    """Query's map (Octree.cpp:322-324, 665): centre and 1/size computed in f32, then widened."""
    mn, mx = np.asarray(root_min, np.float32), np.asarray(root_max, np.float32)
    return ((mn + mx) / np.float32(2)).astype(np.float64), (np.float32(1) / (mx - mn)).astype(np.float64)


def locate(block, xyz):
    """Leaf node index per point (-1 outside the root) and the unit-cube coordinates p."""
    cfg = block["config"]
    centre, inv = root_map(list(cfg.root_min), list(cfg.root_max))
    p = (np.asarray(xyz, np.float64) - centre) * inv
    pf = p.astype(np.float32)
    inside = ((pf >= -0.5) & (pf <= 0.5)).all(1)
    nodes = block["nodes"]
    cur = np.zeros(len(p), np.int64)
    for _ in range(64):
        deg = nodes["deg"][cur]
        todo = inside & (deg == INTERNAL)
        if not todo.any():
            break
        mid = ((nodes["mn"][cur] + nodes["mx"][cur]) / np.float32(2)).astype(np.float64)
        b = (p >= mid).astype(np.int64)
        nxt = nodes["child"][cur].astype(np.int64) + b[:, 0] + 2 * b[:, 1] + 4 * b[:, 2]
        cur = np.where(todo, nxt, cur)
    return np.where(inside, cur, -1), p, inv


def leaf_axes(u, degree, depth):
    """Normalised Legendre values and their first and second derivatives, (3 orders, degree+1, n) per axis of u (n,3)."""
    eye = np.eye(degree + 1)
    nl = np.sqrt((2.0 * np.arange(degree + 1) + 1.0) * 2.0 ** depth)[:, None]
    out = []
    for a in range(3):
        v = L.legval(u[:, a], eye)
        d1 = L.legval(u[:, a], L.legder(eye, 1, axis=0)) if degree >= 1 else np.zeros_like(v)
        d2 = L.legval(u[:, a], L.legder(eye, 2, axis=0)) if degree >= 2 else np.zeros_like(v)
        out.append(np.stack([v, d1, d2]) * nl[None])
    return out


def eval_leaf(c, degree, depth, u):
    """P, dP/du (n,3), d2P/du du (n,6) of leaves of one degree and depth at local u (n,3); c (n, COUNTS[degree]) are the
    points' leaf coefficients. Also the sums of absolute terms of each: (vals, abs sums) as two dicts."""
    lx, ly, lz = leaf_axes(u, degree, depth)
    bi = basis_index(degree)
    ax = [lx[:, bi[:, 0]], ly[:, bi[:, 1]], lz[:, bi[:, 2]]]        # (order, term, n)
    ct = np.asarray(c, np.float64).T                                # (term, n)

    def comp(orders):
        t = ct * ax[0][orders[0]] * ax[1][orders[1]] * ax[2][orders[2]]
        return t.sum(0), np.abs(t).sum(0)

    v, va = comp((0, 0, 0))
    g, ga = np.zeros((len(u), 3)), np.zeros((len(u), 3))
    for a in range(3):
        o = [0, 0, 0]; o[a] = 1
        g[:, a], ga[:, a] = comp(o)
    h, ha = np.zeros((len(u), 6)), np.zeros((len(u), 6))
    for k, (a, b) in enumerate(HESS_AXES):
        o = [0, 0, 0]; o[a] += 1; o[b] += 1
        h[:, k], ha[:, k] = comp(o)
    return dict(value=v, grad=g, hess=h), dict(value=va, grad=ga, hess=ha)


def query_derivatives(block, xyz):
    """The contract for points xyz (n,3) of the tree in `block` (hp.parse_block). Returns (dict value / grad / hess in user
    space, dict of their sums of absolute terms, leaf index per point, local u (n,3))."""
    leaf, p, inv = locate(block, xyz)
    nodes, coeffs = block["nodes"], block["coeffs"]
    n = len(p)
    val = dict(value=np.full(n, DBL_MAX), grad=np.zeros((n, 3)), hess=np.zeros((n, 6)))
    absum = dict(value=np.zeros(n), grad=np.zeros((n, 3)), hess=np.zeros((n, 6)))
    u = np.zeros((n, 3))
    ok = leaf >= 0
    deg = np.where(ok, nodes["deg"][np.maximum(leaf, 0)], -1).astype(np.int64)
    dep = nodes["depth"][np.maximum(leaf, 0)].astype(np.int64)
    mid = ((nodes["mn"][np.maximum(leaf, 0)] + nodes["mx"][np.maximum(leaf, 0)]) / np.float32(2)).astype(np.float64)
    scale = 2.0 ** (dep + 1)
    u[ok] = (p[ok] - mid[ok]) * scale[ok, None]
    s = scale[:, None] * inv[None, :]                               # du_a / dx_a
    for m in np.unique(deg[ok]):
        for d in np.unique(dep[deg == m]):
            sel = np.nonzero((deg == m) & (dep == d))[0]
            cs = nodes["cstart"][leaf[sel]].astype(np.int64)
            c = coeffs[cs[:, None] + np.arange(COUNTS[m])[None, :]]
            r, ra = eval_leaf(c, int(m), int(d), u[sel])
            ss = s[sel]
            hs = np.stack([ss[:, a] * ss[:, b] for a, b in HESS_AXES], 1)
            val["value"][sel], absum["value"][sel] = r["value"], ra["value"]
            val["grad"][sel], absum["grad"][sel] = r["grad"] * ss, ra["grad"] * ss
            val["hess"][sel], absum["hess"][sel] = r["hess"] * hs, ra["hess"] * hs
    return val, absum, leaf, u


def markov(n, k):
    """V. A. Markov's bound: |q^(k)| <= markov(n, k) max|q| on [-1, 1] for a polynomial q of degree n."""
    if k > n:
        return 0.0
    r = 1.0
    for j in range(k):
        r *= (n * n - j * j) / (2.0 * j + 1.0)
    return r
