// isosurface_kernels.cuh — hpsdf_extract_isosurface: the level set F = iso of a tree as a triangle mesh, by marching
// tetrahedra over a uniform grid of Query values.
//
// Grid point (i,j,k) is lo + idx * h per axis (one rounded multiply, then one rounded add: __dmul_rn / __dadd_rn, so nvcc
// cannot contract them into an FMA that a host checker would not reproduce); its linear index is i + (n0+1)(j + (n1+1)k).
// Every cell is cut into the six Kuhn tetrahedra with corners 0, e_a0, e_a0+e_a1, 7 (axis orders xyz, xzy, yxz, yzx, zxy,
// zyx; corner offsets x = bit 0, y = bit 1, z = bit 2). All cells use the same diagonal, so the cut is conforming, and every
// tetrahedron edge joins a grid point q to q + d for a corner offset d in 1..7: q owns that edge. The passes:
//   isoGridKernel   V at every grid point (findLeaf + evalWarp, the path of queryKernel, so V is bitwise hpsdf_query's)
//   isoCountKernel  per point the 7-bit mask of its owned edges that cross (inside = V < iso) and, when the point is a
//                   cell's lowest corner, the inside bits of that cell's eight corners; 64-bit totals of both
//   two exclusive scans (CUB) of popcount(mask) and of the cell's triangle count: vertex and triangle bases
//   isoEmitKernel   one vertex per crossing owned edge, in owner order then d ascending
//   isoTriKernel    the triangles of every cell, in tetrahedron order, with the winding fixed per case (c_isoTet)
#pragma once
#include <cub/cub.cuh>
#include <thrust/iterator/transform_iterator.h>
#include "query_kernels.cuh"

namespace hpsdf
{
    // Triangles of one tetrahedron for one labelling of its chain corners (bit c = chain corner c is inside): count and three
    // edges per triangle, each edge as its owner's corner offset | direction << 3.
    struct IsoTetCase { uint8_t n; uint8_t e[6]; uint8_t pad; };
    __constant__ IsoTetCase c_isoTet[6][16];
    __constant__ uint8_t    c_isoChain[6][4];       // corner offsets of the chain 0, e_a0, e_a0 + e_a1, 7
    __constant__ uint8_t    c_isoCellTris[256];     // triangles of a cell by the inside bits of its eight corners

    // The case tables. One corner alone on its side: one triangle on the edges from it to the other three, in chain order.
    // Two inside corners a < b and two outside c < d (chain positions): (ac, ad, bd) and (ac, bd, bc), always split along
    // ac-bd. The winding then follows from the labels alone: with vertices at the edge midpoints the normal must point from the
    // inside corners to the outside ones; if it does not, the last two vertices of every triangle of the case are swapped.
    inline void isoBuildTables(IsoTetCase tet[6][16], uint8_t chain[6][4], uint8_t cellTris[256])
    {
        static const int order[6][3] = { { 0, 1, 2 }, { 0, 2, 1 }, { 1, 0, 2 }, { 1, 2, 0 }, { 2, 0, 1 }, { 2, 1, 0 } };
        for (int t = 0; t < 6; ++t)
        {
            chain[t][0] = 0;
            chain[t][1] = (uint8_t)(1 << order[t][0]);
            chain[t][2] = (uint8_t)(chain[t][1] | (1 << order[t][1]));
            chain[t][3] = 7;
            for (int L = 0; L < 16; ++L)
            {
                IsoTetCase& cs = tet[t][L];
                cs = IsoTetCase{};
                int in[4], out[4], ni = 0, no = 0;
                for (int c = 0; c < 4; ++c) { if ((L >> c) & 1) in[ni++] = c; else out[no++] = c; }
                int tri[2][3][2], nt = 0;
                if (ni == 1 || ni == 3)
                {
                    const int lone = ni == 1 ? in[0] : out[0];
                    int k = 0;
                    for (int c = 0; c < 4; ++c)
                        if (c != lone) { tri[0][k][0] = lone; tri[0][k][1] = c; ++k; }
                    nt = 1;
                }
                else if (ni == 2)
                {
                    const int a = in[0], b = in[1], c = out[0], d = out[1];
                    const int t0[3][2] = { { a, c }, { a, d }, { b, d } }, t1[3][2] = { { a, c }, { b, d }, { b, c } };
                    for (int v = 0; v < 3; ++v) for (int s = 0; s < 2; ++s) { tri[0][v][s] = t0[v][s]; tri[1][v][s] = t1[v][s]; }
                    nt = 2;
                }
                if (!nt) continue;
                // twice the midpoints, and k_in k_out times (outside centroid - inside centroid): all integers
                auto pos = [&](int c, int a) { return (chain[t][c] >> a) & 1; };
                int m[3][3], dir[3];
                for (int v = 0; v < 3; ++v) for (int a = 0; a < 3; ++a) m[v][a] = pos(tri[0][v][0], a) + pos(tri[0][v][1], a);
                for (int a = 0; a < 3; ++a)
                {
                    int si = 0, so = 0;
                    for (int c = 0; c < ni; ++c) si += pos(in[c], a);
                    for (int c = 0; c < no; ++c) so += pos(out[c], a);
                    dir[a] = ni * so - no * si;
                }
                const int u[3] = { m[1][0] - m[0][0], m[1][1] - m[0][1], m[1][2] - m[0][2] };
                const int w[3] = { m[2][0] - m[0][0], m[2][1] - m[0][1], m[2][2] - m[0][2] };
                const int nrm[3] = { u[1] * w[2] - u[2] * w[1], u[2] * w[0] - u[0] * w[2], u[0] * w[1] - u[1] * w[0] };
                if (nrm[0] * dir[0] + nrm[1] * dir[1] + nrm[2] * dir[2] < 0)
                    for (int k = 0; k < nt; ++k)
                        for (int s = 0; s < 2; ++s) { const int x = tri[k][1][s]; tri[k][1][s] = tri[k][2][s]; tri[k][2][s] = x; }
                cs.n = (uint8_t)nt;
                for (int k = 0; k < nt; ++k)
                    for (int v = 0; v < 3; ++v)
                    {
                        const int lo = chain[t][std::min(tri[k][v][0], tri[k][v][1])], hi = chain[t][std::max(tri[k][v][0], tri[k][v][1])];
                        cs.e[3 * k + v] = (uint8_t)(lo | ((lo ^ hi) << 3));
                    }
            }
        }
        for (int lab = 0; lab < 256; ++lab)
        {
            int n = 0;
            for (int t = 0; t < 6; ++t)
            {
                int L = 0;
                for (int c = 0; c < 4; ++c) L |= ((lab >> chain[t][c]) & 1) << c;
                n += tet[t][L].n;
            }
            cellTris[lab] = (uint8_t)n;
        }
    }

    __device__ __forceinline__ double isoCoord(const IsoGrid& g, int a, uint32_t idx)
    {
        return __dadd_rn(g.lo[a], __dmul_rn((double)idx, g.h[a]));
    }

    // A warp takes 32 consecutive points (mostly one x row, so neighbouring lanes mostly share a leaf); the coordinates are
    // made in registers. Persistent grid with the top table staged once per CTA, as queryKernel.
    __global__ void __launch_bounds__(kQueryThreads, kQueryBlocksPerSm)
    isoGridKernel(const DeviceTreeView view, const IsoGrid g, double* __restrict__ vals)
    {
        __shared__ uint32_t sTop[4096];
        const bool useTop = stageTop(sTop, view.top);
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const uint32_t px = g.n[0] + 1, py = g.n[1] + 1, n = px * py * (g.n[2] + 1);
        const uint32_t nGroups = (n + 31) / 32, warpsTotal = gridDim.x * (kQueryThreads / 32);
        for (uint32_t grp = blockIdx.x * (kQueryThreads / 32) + warp; grp < nGroups; grp += warpsTotal)
        {
            const uint32_t p = grp * 32 + lane;
            LeafHit h;
            if (p < n)
            {
                const uint32_t i = p % px, r = p / px, j = r % py, k = r / py;
                h = findLeaf(view, useTop ? sTop : nullptr, isoCoord(g, 0, i), isoCoord(g, 1, j), isoCoord(g, 2, k));
            }
            const double v = evalWarp(h, view.bidx);
            if (p < n) __stcs(vals + p, v);
        }
    }

    // Persistent grid: the two 64-bit totals take one atomic per CTA.
    __global__ void __launch_bounds__(256)
    isoCountKernel(const IsoGrid g, const double* __restrict__ vals, uint8_t* __restrict__ mask, uint8_t* __restrict__ label,
                   unsigned long long* __restrict__ totals)
    {
        __shared__ uint32_t sV[8], sT[8];
        const uint32_t px = g.n[0] + 1, py = g.n[1] + 1, pxy = px * py, n = pxy * (g.n[2] + 1);
        uint32_t nv = 0, nt = 0;
        for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x)
        {
            const uint32_t i = p % px, r = p / px, j = r % py, k = r / py;
            const bool hx = i < g.n[0], hy = j < g.n[1], hz = k < g.n[2];
            uint32_t in = 0, valid = 0;
            #pragma unroll
            for (int c = 0; c < 8; ++c)
            {
                if (((c & 1) && !hx) || ((c & 2) && !hy) || ((c & 4) && !hz)) continue;
                valid |= 1u << c;
                const uint32_t q = p + (c & 1) + ((c & 2) ? px : 0u) + ((c & 4) ? pxy : 0u);
                if (vals[q] < g.iso) in |= 1u << c;
            }
            uint32_t m = 0;
            #pragma unroll
            for (int d = 1; d < 8; ++d)
                if (((valid >> d) & 1) && ((in >> d) & 1) != (in & 1)) m |= 1u << (d - 1);
            const uint32_t lab = (hx && hy && hz) ? in : 0u;          // label 0 (all outside) has no triangles
            mask[p] = (uint8_t)m;
            label[p] = (uint8_t)lab;
            nv += __popc(m);
            nt += c_isoCellTris[lab];
        }
        nv = __reduce_add_sync(0xFFFFFFFFu, nv);
        nt = __reduce_add_sync(0xFFFFFFFFu, nt);
        if ((threadIdx.x & 31) == 0) { sV[threadIdx.x >> 5] = nv; sT[threadIdx.x >> 5] = nt; }
        __syncthreads();
        if (threadIdx.x == 0)
        {
            unsigned long long a = 0, b = 0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { a += sV[w]; b += sT[w]; }
            if (a) atomicAdd(totals, a);
            if (b) atomicAdd(totals + 1, b);
        }
    }

    struct IsoPopc { __device__ uint32_t operator()(uint8_t m) const { return (uint32_t)__popc(m); } };
    struct IsoCellTriCount
    {
        __device__ uint32_t operator()(uint8_t lab) const { return c_isoCellTris[lab]; }
    };

    // t = (iso - V(q)) / (V(q+d) - V(q)), x = P(q) + t (P(q+d) - P(q)): each operation correctly rounded in f64, then one
    // rounding to f32.
    __global__ void __launch_bounds__(256)
    isoEmitKernel(const IsoGrid g, const double* __restrict__ vals, const uint8_t* __restrict__ mask, const uint32_t* __restrict__ vbase,
                  float* __restrict__ verts)
    {
        const uint32_t px = g.n[0] + 1, py = g.n[1] + 1, pxy = px * py, n = pxy * (g.n[2] + 1);
        const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
        if (p >= n) return;
        const uint32_t m = mask[p];
        if (!m) return;
        const uint32_t idx[3] = { p % px, (p / px) % py, p / pxy };
        const double v0 = vals[p];
        const double x0[3] = { isoCoord(g, 0, idx[0]), isoCoord(g, 1, idx[1]), isoCoord(g, 2, idx[2]) };
        size_t o = vbase[p];
        for (int d = 1; d < 8; ++d)
        {
            if (!((m >> (d - 1)) & 1)) continue;
            const uint32_t q = p + (d & 1) + ((d & 2) ? px : 0u) + ((d & 4) ? pxy : 0u);
            const double t = __ddiv_rn(__dsub_rn(g.iso, v0), __dsub_rn(vals[q], v0));
            #pragma unroll
            for (int a = 0; a < 3; ++a)
            {
                const double x1 = ((d >> a) & 1) ? isoCoord(g, a, idx[a] + 1) : x0[a];
                verts[3 * o + a] = __double2float_rn(__dadd_rn(x0[a], __dmul_rn(t, __dsub_rn(x1, x0[a]))));
            }
            ++o;
        }
    }

    __global__ void __launch_bounds__(256)
    isoTriKernel(const IsoGrid g, const uint8_t* __restrict__ label, const uint8_t* __restrict__ mask, const uint32_t* __restrict__ vbase,
                 const uint32_t* __restrict__ tbase, uint32_t* __restrict__ tris)
    {
        const uint32_t px = g.n[0] + 1, pxy = px * (g.n[1] + 1), n = pxy * (g.n[2] + 1);
        const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
        if (p >= n) return;
        const uint32_t lab = label[p];
        if (lab == 0 || lab == 0xFF) return;
        size_t o = tbase[p];
        for (int t = 0; t < 6; ++t)
        {
            uint32_t L = 0;
            #pragma unroll
            for (int c = 0; c < 4; ++c) L |= ((lab >> c_isoChain[t][c]) & 1u) << c;
            const IsoTetCase cs = c_isoTet[t][L];
            for (int e = 0; e < 3 * cs.n; ++e)
            {
                const uint32_t off = cs.e[e] & 7, d = cs.e[e] >> 3;
                const uint32_t q = p + (off & 1) + ((off & 2) ? px : 0u) + ((off & 4) ? pxy : 0u);
                tris[3 * o + e] = vbase[q] + __popc(mask[q] & ((1u << (d - 1)) - 1u));
            }
            o += cs.n;
        }
    }
}
