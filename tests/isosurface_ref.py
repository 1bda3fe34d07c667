"""Numpy restatement of the contract of hpsdf_extract_isosurface (include/hpsdf.h, DESIGN.md §11), bit for bit, and the mesh
checks the isosurface tests use. Vectorised over grid points and over the cells the surface passes through."""
import numpy as np

# axis orders xyz, xzy, yxz, yzx, zxy, zyx -> Kuhn chains 0, e_a0, e_a0 + e_a1, 7 (corner offsets: x = 1, y = 2, z = 4)
ORDERS = [(0, 1, 2), (0, 2, 1), (1, 0, 2), (1, 2, 0), (2, 0, 1), (2, 1, 0)]
CHAINS = [(0, 1 << a, (1 << a) | (1 << b), 7) for a, b, _ in ORDERS]


def _corner(o):
    return np.array([o & 1, (o >> 1) & 1, (o >> 2) & 1], np.float64)


def tet_cases():
    """cases[t][L]: the triangles of tetrahedron t when chain corner c is inside iff bit c of L is set; each triangle is
    three edges (owner corner offset, direction)."""
    cases = []
    for ch in CHAINS:
        row = []
        for L in range(16):
            ins = [c for c in range(4) if (L >> c) & 1]
            outs = [c for c in range(4) if not (L >> c) & 1]
            if len(ins) in (1, 3):
                lone = ins[0] if len(ins) == 1 else outs[0]
                tris = [[(lone, c) for c in range(4) if c != lone]]
            elif len(ins) == 2:
                (a, b), (c, d) = ins, outs
                tris = [[(a, c), (a, d), (b, d)], [(a, c), (b, d), (b, c)]]
            else:
                tris = []
            if tris:
                mid = [(_corner(ch[x]) + _corner(ch[y])) / 2 for x, y in tris[0]]
                nrm = np.cross(mid[1] - mid[0], mid[2] - mid[0])
                towards_out = np.mean([_corner(ch[c]) for c in outs], 0) - np.mean([_corner(ch[c]) for c in ins], 0)
                if nrm @ towards_out < 0:
                    tris = [[t[0], t[2], t[1]] for t in tris]
            row.append([[(ch[min(x, y)], ch[min(x, y)] ^ ch[max(x, y)]) for x, y in t] for t in tris])
        cases.append(row)
    return cases


def grid_axes(n, lo, hi):
    """Coordinates of the grid points along each axis: lo + idx * h, one rounded multiply and one rounded add."""
    out = []
    for a in range(3):
        h = (np.float64(hi[a]) - np.float64(lo[a])) / np.float64(n[a])
        out.append(np.float64(lo[a]) + np.arange(n[a] + 1, dtype=np.float64) * h)
    return out


def grid_points(n, lo, hi):
    """All grid points, (N, 3) f64, in linear order i + (n0+1)(j + (n1+1)k)."""
    xs, ys, zs = grid_axes(n, lo, hi)
    Z, Y, X = np.meshgrid(zs, ys, xs, indexing="ij")
    return np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1)


def extract(vals, n, lo, hi, iso):
    """The mesh of the contract from the grid values (linear order) -> (vertices (V,3) f32, triangles (T,3) u32)."""
    n0, n1, n2 = (int(x) for x in n)
    px, py, pz = n0 + 1, n1 + 1, n2 + 1
    vals = np.asarray(vals, np.float64).ravel()
    inside = (vals < iso).reshape(pz, py, px)
    cross = np.zeros((pz, py, px, 7), bool)
    for d in range(1, 8):
        dx, dy, dz = d & 1, (d >> 1) & 1, (d >> 2) & 1
        cross[:pz - dz, :py - dy, :px - dx, d - 1] = inside[:pz - dz, :py - dy, :px - dx] != inside[dz:, dy:, dx:]
    cross = cross.reshape(-1, 7)
    owner, dm1 = np.nonzero(cross)                       # owner order, then d ascending
    d = dm1 + 1
    idx = [owner % px, (owner // px) % py, owner // (px * py)]
    q = owner + (d & 1) + ((d >> 1) & 1) * px + ((d >> 2) & 1) * px * py
    v0 = vals[owner]
    t = (iso - v0) / (vals[q] - v0)
    axes = grid_axes(n, lo, hi)
    verts = np.empty((len(owner), 3), np.float32)
    for a in range(3):
        x0 = axes[a][idx[a]]
        x1 = axes[a][idx[a] + ((d >> a) & 1)]
        verts[:, a] = (x0 + t * (x1 - x0)).astype(np.float32)
    counts = cross.sum(1)
    vbase = np.cumsum(counts) - counts
    before = np.cumsum(cross, 1) - cross                 # crossing edges of the owner with a smaller direction

    # cells: inside bits of the eight corners; only mixed cells have triangles
    label = np.zeros((n2, n1, n0), np.int64)
    for c in range(8):
        dx, dy, dz = c & 1, (c >> 1) & 1, (c >> 2) & 1
        label |= inside[dz:dz + n2, dy:dy + n1, dx:dx + n0].astype(np.int64) << c
    label = label.ravel()
    cells = np.nonzero((label != 0) & (label != 255))[0]  # ascending cell index = ascending lowest-corner point index
    ci, cj, ck = cells % n0, (cells // n0) % n1, cells // (n0 * n1)
    P = ci + px * (cj + py * ck)
    lab = label[cells]
    cases = tet_cases()
    ntri = np.zeros((6, 16), np.int64)
    code = np.zeros((6, 16, 2, 3), np.int64)
    for tt in range(6):
        for L in range(16):
            ntri[tt, L] = len(cases[tt][L])
            for s, tri in enumerate(cases[tt][L]):
                for v, (off, dd) in enumerate(tri):
                    code[tt, L, s, v] = off | (dd << 3)
    out = np.zeros((len(cells), 6, 2, 3), np.int64)
    valid = np.zeros((len(cells), 6, 2), bool)
    for tt, ch in enumerate(CHAINS):
        L = sum(((lab >> ch[c]) & 1) << c for c in range(4))
        for s in range(2):
            valid[:, tt, s] = ntri[tt, L] > s
            for v in range(3):
                e = code[tt, L, s, v]
                off, dd = e & 7, e >> 3
                qq = P + (off & 1) + ((off >> 1) & 1) * px + ((off >> 2) & 1) * px * py
                out[:, tt, s, v] = np.where(valid[:, tt, s], vbase[qq] + before[qq, np.maximum(dd, 1) - 1], 0)
    tris = out[valid].astype(np.uint32)
    return verts, tris


def canonical_rows(tris):
    """Each triangle rotated so that its smallest index comes first (a rotation keeps the orientation)."""
    t = np.asarray(tris, np.int64).reshape(-1, 3)
    r = np.argmin(t, 1)
    return np.stack([t[np.arange(len(t)), (r + k) % 3] for k in range(3)], 1)


def mesh_report(verts, tris):
    """closed_oriented: every directed edge appears once and its reverse once; all_used: every vertex is in a triangle;
    euler: V - E + F; volume: signed volume (positive when triangles are counter-clockwise seen from outside)."""
    t = np.asarray(tris, np.int64).reshape(-1, 3)
    nv = len(verts)
    a = np.concatenate([t[:, 0], t[:, 1], t[:, 2]])
    b = np.concatenate([t[:, 1], t[:, 2], t[:, 0]])
    key = a * nv + b
    uniq, cnt = np.unique(key, return_counts=True)
    closed = bool(len(t)) and bool((cnt == 1).all()) and bool(np.isin(b * nv + a, uniq).all())
    und = np.unique(np.minimum(a, b) * nv + np.maximum(a, b))
    used = np.zeros(nv, bool)
    used[t.ravel()] = True
    v = np.asarray(verts, np.float64)
    vol = float(np.einsum("ij,ij->i", v[t[:, 0]], np.cross(v[t[:, 1]], v[t[:, 2]])).sum() / 6.0) if len(t) else 0.0
    return dict(closed_oriented=closed, all_used=bool(used.all()), euler=int(nv - len(und) + len(t)), volume=vol)
