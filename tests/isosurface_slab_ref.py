"""Plane-by-plane torch restatement of the contract of hpsdf_extract_isosurface (DESIGN.md §11), bit for bit, for grids
too large for isosurface_ref.extract. It holds the values of three z-planes at a time and running 64-bit vertex and
triangle bases; values come from a callable, so the same code runs on a numpy field on the CPU and on hpsdf_query_device
on the GPU. It shares no code with the kernels (the case tables come from isosurface_ref.tet_cases)."""
import numpy as np
import torch

from isosurface_ref import CHAINS, tet_cases


def _axes(n, lo, hi, device):
    out = []
    for a in range(3):
        h = (float(hi[a]) - float(lo[a])) / float(n[a])
        idx = torch.arange(n[a] + 1, dtype=torch.float64, device=device)
        out.append(torch.mul(idx, h).add(float(lo[a])))        # one rounded multiply, then one rounded add: nothing fuses
    return out


def _case_codes(device):
    cases = tet_cases()
    ntri = torch.zeros((6, 16), dtype=torch.int64)
    code = torch.zeros((6, 16, 2, 3), dtype=torch.int64)
    for t in range(6):
        for L in range(16):
            ntri[t, L] = len(cases[t][L])
            for s, tri in enumerate(cases[t][L]):
                for v, (off, d) in enumerate(tri):
                    code[t, L, s, v] = off | (d << 3)
    return ntri.to(device), code.to(device)


def extract(values, n, lo, hi, iso, device="cpu"):
    """values(points (m,3) f64 tensor) -> (m,) f64 tensor. Returns (vertices (V,3) float32, triangles (T,3) int64) as
    tensors on `device`."""
    n0, n1, n2 = (int(x) for x in n)
    px, py = n0 + 1, n1 + 1
    xs, ys, zs = _axes((n0, n1, n2), lo, hi, device)
    X, Y = xs[None, :].expand(py, px), ys[:, None].expand(py, px)
    ntri, code = _case_codes(device)

    def plane_values(k):
        P = torch.stack([X.reshape(-1), Y.reshape(-1), zs[k].expand(py * px)], 1).contiguous()
        return values(P).reshape(py, px)

    def plane_edges(ins, ins_up):
        """(py, px, 7) crossing owned edges of a plane's points; ins_up: the inside flags of the next plane or None."""
        cross = torch.zeros((py, px, 7), dtype=torch.bool, device=device)
        for d in range(1, 8):
            dx, dy, dz = d & 1, (d >> 1) & 1, (d >> 2) & 1
            if dz and ins_up is None:
                continue
            far = ins_up if dz else ins
            cross[:py - dy, :px - dx, d - 1] = ins[:py - dy, :px - dx] != far[dy:, dx:]
        return cross

    verts, tris = [], []
    vrun = 0
    vals = plane_values(0)
    nxt = plane_values(1) if n2 >= 1 else None
    prev = None                                            # (inside, vbase, before) of the plane below
    for k in range(n2 + 1):
        ins = vals < iso
        ins_up = nxt < iso if nxt is not None else None
        cross = plane_edges(ins, ins_up)
        counts = cross.sum(2).reshape(-1)
        vbase = (torch.cumsum(counts, 0) - counts + vrun).reshape(py, px)
        before = torch.cumsum(cross.to(torch.int64), 2) - cross.to(torch.int64)
        j, i, dm1 = torch.nonzero(cross, as_tuple=True)     # owner order, then d
        d = dm1 + 1
        dx, dy, dz = d & 1, (d >> 1) & 1, (d >> 2) & 1
        v0 = vals[j, i]
        v1 = torch.where(dz.bool(), nxt[j + dy, i + dx] if nxt is not None else v0, vals[j + dy, i + dx])
        t = torch.div(iso - v0, torch.sub(v1, v0))
        kk = torch.full_like(i, k)
        cols = []
        for ax, idx, step in ((xs, i, dx), (ys, j, dy), (zs, kk, dz)):
            x0, x1 = ax[idx], ax[idx + step]
            cols.append(torch.add(x0, torch.mul(t, torch.sub(x1, x0))).to(torch.float32))
        verts.append(torch.stack(cols, 1))
        vrun += int(counts.sum())
        if prev is not None:                               # cells of layer k - 1: corners on planes k - 1 and k
            planes = (prev, (ins, vbase, before))
            label = torch.zeros((n1, n0), dtype=torch.int64, device=device)
            for c in range(8):
                cx, cy, cz = c & 1, (c >> 1) & 1, (c >> 2) & 1
                label |= planes[cz][0][cy:cy + n1, cx:cx + n0].to(torch.int64) << c
            cj, ci = torch.nonzero((label != 0) & (label != 255), as_tuple=True)
            lab = label[cj, ci]
            out = torch.zeros((len(ci), 6, 2, 3), dtype=torch.int64, device=device)
            valid = torch.zeros((len(ci), 6, 2), dtype=torch.bool, device=device)
            for tt, ch in enumerate(CHAINS):
                L = sum(((lab >> ch[c]) & 1) << c for c in range(4))
                for s in range(2):
                    valid[:, tt, s] = ntri[tt, L] > s
                    for v in range(3):
                        e = code[tt, L, s, v]
                        off, dd = e & 7, e >> 3
                        qi, qj, qz = ci + (off & 1), cj + ((off >> 1) & 1), (off >> 2) & 1
                        dd1 = torch.clamp(dd, min=1) - 1
                        got = torch.zeros_like(ci)
                        for z in (0, 1):
                            vb, bf = planes[z][1], planes[z][2]
                            sel = qz == z
                            got = torch.where(sel, vb[qj.clamp(max=py - 1), qi.clamp(max=px - 1)] +
                                              bf[qj.clamp(max=py - 1), qi.clamp(max=px - 1), dd1], got)
                        out[:, tt, s, v] = torch.where(valid[:, tt, s], got, torch.zeros_like(got))
            tris.append(out[valid])
        prev = (ins, vbase, before)
        vals, nxt = nxt, (plane_values(k + 2) if k + 2 <= n2 else None)
    V = torch.cat(verts) if verts else torch.empty((0, 3), dtype=torch.float32, device=device)
    T = torch.cat(tris) if tris else torch.empty((0, 3), dtype=torch.int64, device=device)
    return V, T.reshape(-1, 3)


def numpy_field(f):
    """A values callable from a numpy field f((m,3) f64 array) -> (m,) f64 array."""
    return lambda P: torch.from_numpy(np.ascontiguousarray(f(P.cpu().numpy()), np.float64)).to(P.device)


def query_field(tree):
    """A values callable from hpsdf_query_device on the current stream of the tensor's device."""
    return lambda P: tree.QueryTorch(P.contiguous())
