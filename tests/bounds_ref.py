"""Checker of the hpsdf_query_bounds contract (DESIGN §14). It shares no code with the kernel: leaves come from the
MemoryBlock (cell = the node's f32 box, degree, depth, coefficients), the participating leaves from a vectorised test of
every leaf's extended cell against the box, and each leaf's Bernstein coefficients by another route than the kernel's
collocation: per axis, the exact monomial form of each normalised Legendre polynomial is re-expanded about the centre of the
clipped interval and converted to the degree-p Bernstein basis in mpmath at 40 digits; the three axes are contracted in
80-bit long double, whose rounding (below 1e-13 of S_leaf even at degree 12) is far inside the allowance. kappa_p is derived
here from its formula (DESIGN §14), with the inverse collocation norms computed in mpmath."""
from fractions import Fraction
from functools import lru_cache
from math import comb

import mpmath as mp
import numpy as np

INTERNAL = 13
COUNTS = [1, 4, 10, 20, 35, 56, 83, 120, 165, 220, 286, 364, 455]
DBL_MAX = np.finfo(np.float64).max
L = 0.5 + 2.0 ** -25            # |p| <= L: the f32 cast of p lies in [-0.5, 0.5]
LD = np.longdouble
mp.mp.dps = 40


def basis_index(degree):
    """(a, b, c) Legendre degrees of x, y, z per coefficient: shell by shell, a then b, c = p - a - b; 83 at degree 6."""
    out = [(a, b, p - a - b) for p in range(degree + 1) for a in range(p + 1) for b in range(p - a + 1)]
    return np.array(out[:COUNTS[degree]], np.int64)


def root_map(root_min, root_max):
    """Query's map: centre and 1/size computed in f32, then widened."""
    mn, mx = np.asarray(root_min, np.float32), np.asarray(root_max, np.float32)
    return ((mn + mx) / np.float32(2)).astype(np.float64), (np.float32(1) / (mx - mn)).astype(np.float64)


@lru_cache(None)
def collocation_norm(p):
    """||C_p^-1||_inf of the Bernstein collocation matrix at the Chebyshev-Lobatto nodes sin^2(pi j / 2p) of [0, 1]."""
    if p == 0:
        return mp.mpf(1)
    tau = [mp.sin(mp.pi * j / (2 * p)) ** 2 for j in range(p + 1)]
    c = mp.matrix(p + 1, p + 1)
    for j in range(p + 1):
        for i in range(p + 1):
            c[j, i] = comb(p, i) * tau[j] ** i * (1 - tau[j]) ** (p - i)
    ci = c ** -1
    return max(sum(abs(ci[r, k]) for k in range(p + 1)) for r in range(p + 1))


@lru_cache(None)
def kappa_log2(p):
    """log2 kappa_p = ceil(log2(G^3 (Q_p + 3 W_p E_p + (3p + 4) W_p))), G = 1.01, Q_p = 36 p^2 + n_p + 5,
    W_p = binom(p, p // 2), E_p = ||C_p^-1|| (15 p^2 + 4 p + 3) (DESIGN §14)."""
    w = comb(p, p // 2)
    e = collocation_norm(p) * (15 * p * p + 4 * p + 3)
    total = mp.mpf("1.01") ** 3 * (36 * p * p + COUNTS[p] + 5 + 3 * w * e + (3 * p + 4) * w)
    return int(mp.ceil(mp.log(total, 2)))


@lru_cache(None)
def legendre_monomial(j):
    """Exact monomial coefficients of P_j (low to high)."""
    out = [Fraction(0)] * (j + 1)
    for k in range(j // 2 + 1):
        out[j - 2 * k] = Fraction((-1) ** k * comb(j, k) * comb(2 * j - 2 * k, j), 2 ** j)
    return out


def nl(j, depth):
    return mp.sqrt(mp.mpf((2 * int(j) + 1) * 2 ** int(depth)))


@lru_cache(None)
def axis_matrix(p, depth, ua, ub):
    """M[j][k]: degree-p Bernstein coefficient k of N_j = nl_j P_j on [ua, ub] (mpmath, returned as long double)."""
    a, b = mp.mpf(ua), mp.mpf(ub)
    m, w = (a + b) / 2, b - a
    out = np.zeros((p + 1, p + 1), LD)
    for j in range(p + 1):
        mono = [mp.mpf(x.numerator) / x.denominator for x in legendre_monomial(j)]
        # about the centre: q(s) = P_j(m + s)
        d = [mp.fsum(mono[i] * comb(i, k) * m ** (i - k) for i in range(k, j + 1)) for k in range(j + 1)]
        # s = -w/2 + w t, t in [0, 1]
        e = [mp.mpf(0)] * (p + 1)
        for i, di in enumerate(d):
            for k in range(i + 1):
                e[k] += di * comb(i, k) * w ** k * (-w / 2) ** (i - k)
        s = nl(j, depth)
        for r in range(p + 1):
            out[j, r] = LD(str(s * mp.fsum(mp.mpf(comb(r, k)) / comb(p, k) * e[k] for k in range(r + 1))))
    return out


def leaf_poly(coeffs, degree, depth, u):
    """The leaf polynomial at local u (n, 3), in long double."""
    bi = basis_index(degree)
    from numpy.polynomial import legendre as Lg
    eye = np.eye(degree + 1)
    nlv = np.array([float(nl(j, depth)) for j in range(degree + 1)])[:, None]
    ax = [Lg.legval(np.asarray(u[:, a], np.float64), eye) * nlv for a in range(3)]
    t = np.asarray(coeffs, np.float64)[:, None] * ax[0][bi[:, 0]] * ax[1][bi[:, 1]] * ax[2][bi[:, 2]]
    return t.sum(0)


class Leaves:
    """Leaves of a tree: integer cells, depths, degrees, coefficients, and Query's root map."""

    def __init__(self, cells, depth, deg, coeffs, centre=(0.0, 0.0, 0.0), inv=(1.0, 1.0, 1.0)):
        self.cell = np.asarray(cells, np.int64)
        self.depth = np.asarray(depth, np.int64)
        self.deg = np.asarray(deg, np.int64)
        self.coeffs = list(coeffs)
        self.centre, self.inv = np.asarray(centre, np.float64), np.asarray(inv, np.float64)
        size = 2.0 ** -self.depth[:, None]
        lo = self.cell * size - 0.5
        self.c = lo + 0.5 * size
        self.elo = np.where(self.cell == 0, -L, lo)
        self.ehi = np.where(self.cell + 1 == 2 ** self.depth[:, None], L, lo + size)
        self.s = [mp.fsum(abs(mp.mpf(float(c))) * nl(a, dp) * nl(b, dp) * nl(cc, dp) for c, (a, b, cc) in zip(cs, basis_index(int(dg))))
                  for cs, dg, dp in zip(self.coeffs, self.deg, self.depth)]
        self._cell_iv = {}

    @classmethod
    def from_block(cls, blk):
        nodes = blk["nodes"]
        idx = np.nonzero(nodes["deg"] != INTERNAL)[0]
        depth = nodes["depth"][idx].astype(np.int64)
        cells = np.rint((nodes["mn"][idx].astype(np.float64) + 0.5) * 2.0 ** depth[:, None]).astype(np.int64)
        deg = nodes["deg"][idx].astype(np.int64)
        co = [blk["coeffs"][int(nodes["cstart"][i]):int(nodes["cstart"][i]) + COUNTS[int(nodes["deg"][i])]] for i in idx]
        cfg = blk["config"]
        centre, inv = root_map(list(cfg.root_min), list(cfg.root_max))
        out = cls(cells, depth, deg, co, centre, inv)
        out.node = idx
        return out

    def allowance(self, i):
        return float(mp.ldexp(self.s[i], kappa_log2(int(self.deg[i])) - 53))

    def hull(self, i, lo, hi):
        """(min, max) of the exact Bernstein coefficients of leaf i over the unit-cube box [lo, hi] (inside E(leaf))."""
        p, dp = int(self.deg[i]), int(self.depth[i])
        scale = float(2 << dp)
        ua = (np.asarray(lo, np.float64) - self.c[i]) * scale          # the kernel's operations, in f64
        ub = (np.asarray(hi, np.float64) - self.c[i]) * scale
        m = [axis_matrix(p, dp, float(ua[a]), float(ub[a])) for a in range(3)]
        t = np.zeros((p + 1,) * 3, LD)
        for c, (a, b, cc) in zip(self.coeffs[i], basis_index(p)):
            t[a, b, cc] = LD(float(c))
        bern = np.einsum("abc,ak,bl,cm->klm", t, m[0], m[1], m[2], optimize=True)
        return float(bern.min()), float(bern.max()), bern

    def interval(self, i, lo, hi):
        """The contract's interval of leaf i over [lo, hi]: hull widened by A_leaf, intersected with the whole-cell interval."""
        a = self.allowance(i)
        if i not in self._cell_iv:
            mn, mx, _ = self.hull(i, self.elo[i], self.ehi[i])
            self._cell_iv[i] = (mn - a, mx + a)
        ce = self._cell_iv[i]
        if (np.asarray(lo) <= self.elo[i]).all() and (np.asarray(hi) >= self.ehi[i]).all():
            return ce, a
        mn, mx, _ = self.hull(i, lo, hi)
        return (max(mn - a, ce[0]), min(mx + a, ce[1])), a

    def bounds(self, box_lo, box_hi):
        """(f_lo, f_hi, tolerance of f_lo, tolerance of f_hi) of one box in user space."""
        box_lo, box_hi = np.asarray(box_lo, np.float64), np.asarray(box_hi, np.float64)
        if np.isnan(box_lo).any() or np.isnan(box_hi).any() or (box_lo > box_hi).any():
            return np.nan, np.nan, 0.0, 0.0
        with np.errstate(invalid="ignore", over="ignore"):
            plo = (box_lo - self.centre) * self.inv
            phi = (box_hi - self.centre) * self.inv
        if (phi < -L).any() or (plo > L).any():
            return DBL_MAX, DBL_MAX, 0.0, 0.0
        partial = (plo < -L).any() or (phi > L).any()
        hit = np.nonzero(((self.ehi >= plo) & (self.elo <= phi)).all(1))[0]
        ivs = []
        for i in hit:
            (lo, hi), a = self.interval(i, np.maximum(plo, self.elo[i]), np.minimum(phi, self.ehi[i]))
            ivs.append((lo, hi, a))
        ivs = np.array(ivs)
        f_lo, f_hi = ivs[:, 0].min(), ivs[:, 1].max()
        amax = ivs[:, 2].max()
        tol_lo = ivs[ivs[:, 0] <= f_lo + amax + ivs[:, 2], 2].max()
        tol_hi = ivs[ivs[:, 1] >= f_hi - amax - ivs[:, 2], 2].max()
        if partial:
            f_hi, tol_hi = DBL_MAX, 0.0
        return f_lo, f_hi, tol_lo, tol_hi
