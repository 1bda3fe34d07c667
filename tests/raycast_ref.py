"""Numpy checker of the hpsdf_raycast contract (DESIGN §12). It shares neither the kernel's leaf walk nor its root finder:
sub-intervals come from slab tests of the unit-cube ray against every leaf box, sorted by entry; the field on each is sampled
through a caller-given evaluator (tree.Query for real trees) at 2(p+1) interior Chebyshev points, fitted by a degree-p
Chebyshev series whose residual must be at rounding level, and solved with numpy's companion-matrix roots."""
import numpy as np
from numpy.polynomial import chebyshev as Ch

INTERNAL = 13


def root_map(root_min, root_max):
    """Query's map (Octree.cpp:322-324, 665): centre and 1/size computed in f32, then widened."""
    mn, mx = np.asarray(root_min, np.float32), np.asarray(root_max, np.float32)
    centre = ((mn + mx) / np.float32(2)).astype(np.float64)
    inv = (np.float32(1) / (mx - mn)).astype(np.float64)
    return centre, inv


def tree_leaves(block):
    """Leaf boxes (unit cube, f64) and degrees of a parsed MemoryBlock (hp.parse_block)."""
    nodes = block["nodes"]
    leaf = nodes["deg"] != INTERNAL
    return nodes["mn"][leaf].astype(np.float64), nodes["mx"][leaf].astype(np.float64), nodes["deg"][leaf].astype(np.int64)


def clip(p0, dp, t_min, t_max):
    """[ta, tb] of one unit-cube ray inside [-0.5, 0.5]^3, or None."""
    ta, tb = t_min, t_max
    for a in range(3):
        if dp[a] == 0.0:
            if not -0.5 <= p0[a] <= 0.5:
                return None
            continue
        t1, t2 = (-0.5 - p0[a]) / dp[a], (0.5 - p0[a]) / dp[a]
        ta, tb = max(ta, min(t1, t2)), min(tb, max(t1, t2))
    return (ta, tb) if ta <= tb else None


def sub_intervals(p0, dp, ta, tb, lo, hi):
    """Leaves the segment [ta, tb] passes through with a positive length, sorted by entry: (index, enter, exit)."""
    enter = np.full(len(lo), ta)
    leave = np.full(len(lo), tb)
    ok = np.ones(len(lo), bool)
    for a in range(3):
        if dp[a] == 0.0:               # Query's p >= c: a coordinate on a face belongs to the upper cell (or to the root's top)
            ok &= (lo[:, a] <= p0[a]) & ((p0[a] < hi[:, a]) | (hi[:, a] == 0.5))
            continue
        t1, t2 = (lo[:, a] - p0[a]) / dp[a], (hi[:, a] - p0[a]) / dp[a]
        enter = np.maximum(enter, np.minimum(t1, t2))
        leave = np.minimum(leave, np.maximum(t1, t2))
    ok &= leave > enter
    idx = np.nonzero(ok)[0]
    idx = idx[np.argsort(enter[idx], kind="stable")]
    return [(int(i), float(enter[i]), float(leave[i])) for i in idx]


def _segment_min(c, lo_x, hi_x):
    """Minimum of the Chebyshev series c on [lo_x, hi_x] (endpoints and real critical points)."""
    xs = [lo_x, hi_x]
    if len(c) > 2:
        r = Ch.chebroots(Ch.chebder(c))
        xs += [x.real for x in r if abs(x.imag) <= 1e-7 and lo_x <= x.real <= hi_x]
    return min(Ch.chebval(np.array(xs), c))


def cast(o, d, root_min, root_max, lo, hi, deg, evaluate, t_min=0.0, t_max=np.inf, iso=0.0, scale=1.0, tol=1e-11):
    """First crossings of F = iso for rays o + t d. evaluate(points (k,3) user space) -> F. Returns a dict of arrays:
    t (inf for a miss), flag (0 = decided, 1 = near-tangent crossing or near-touch before the hit / within tol*scale of iso,
    2 = a fit residual above rounding level: the leaf of the sampled points is ambiguous), leaves (sub-intervals looked at),
    degrees (list per ray of the leaf degrees in order, up to the hit), at_entry."""
    centre, inv = root_map(root_min, root_max)
    o, d = np.asarray(o, np.float64).reshape(-1, 3), np.asarray(d, np.float64).reshape(-1, 3)
    n = len(o)
    out_t, flag, leaves, degrees = np.full(n, np.inf), np.zeros(n, np.int64), np.zeros(n, np.int64), [[] for _ in range(n)]
    at_entry = np.zeros(n, bool)          # the hit is the start of its sub-interval (a ray starting inside, or a jump at a face)
    tol_g = tol * scale
    # every sub-interval's sample points first, in one evaluator call
    jobs = []
    for r in range(n):
        p0, dp = (o[r] - centre) * inv, d[r] * inv
        if not (np.isfinite(p0).all() and np.isfinite(dp).all()) or not dp.any():
            continue
        c = clip(p0, dp, t_min, t_max)
        if c is None:
            continue
        jobs.append((r, sub_intervals(p0, dp, c[0], c[1], lo, hi)))
    pts, offs, total = [], [], 0
    for r, subs in jobs:
        for k, te, tx in subs:
            m = 2 * (int(deg[k]) + 1)
            x = np.cos(np.pi * (np.arange(m) + 0.5) / m)
            t = te + (x + 1.0) * 0.5 * (tx - te)
            offs.append(total)
            total += m
            pts.append(o[r][None, :] + t[:, None] * d[r][None, :])
    vals = evaluate(np.concatenate(pts)) if pts else np.empty(0)
    j = 0
    for r, subs in jobs:
        done = False
        for k, te, tx in subs:
            p = int(deg[k])
            m = 2 * (p + 1)
            if done:
                j += 1
                continue
            x = np.cos(np.pi * (np.arange(m) + 0.5) / m)
            v = vals[offs[j]:offs[j] + m] - iso
            j += 1
            leaves[r] += 1
            degrees[r].append(p)
            c = Ch.chebfit(x, v, p)
            if np.abs(Ch.chebval(x, c) - v).max() > 1e-12 * max(np.abs(v).max(), scale):
                flag[r] = 2
                done = True
                continue
            g0 = Ch.chebval(-1.0, c)
            if g0 <= 0.0:
                out_t[r] = te
                at_entry[r] = True
                if g0 > -tol_g:
                    flag[r] = 1
                done = True
                continue
            top = np.abs(c).max()
            while len(c) > 1 and abs(c[-1]) <= 1e-15 * top:     # a lower-degree restriction: drop the rounding-level tail
                c = c[:-1]
            roots = [x_.real for x_ in (Ch.chebroots(c) if len(c) > 1 else []) if abs(x_.imag) <= 1e-7 and -1.0 <= x_.real <= 1.0]
            hit_x = min(roots) if roots else None
            seg_min = _segment_min(c, -1.0, hit_x if hit_x is not None else 1.0)
            if hit_x is None:
                if seg_min <= tol_g:
                    flag[r] = 1                      # a near-touch that rounding may turn into a hit
                continue
            out_t[r] = te + (hit_x + 1.0) * 0.5 * (tx - te)
            slope = abs(Ch.chebval(hit_x, Ch.chebder(c))) * 2.0 / (tx - te)       # |dg/dt|
            dt = tol_g / slope if slope > 0 else np.inf
            # near-touch before the hit, or a crossing so flat that rounding of g moves it by more than 1e-10 of `scale`
            near_before = _segment_min(c, -1.0, max(-1.0, hit_x - 1e-6)) <= tol_g if hit_x > -1.0 + 1e-6 else False
            if near_before or dt * np.linalg.norm(d[r]) > 1e-10 * scale:
                flag[r] = 1
            done = True
    return dict(t=out_t, flag=flag, leaves=leaves, degrees=degrees, at_entry=at_entry)
