// isosurface_sparse_kernels.cuh — hpsdf_extract_isosurface_sparse: the mesh of hpsdf_extract_isosurface (same grid, values,
// tetrahedra, vertex and triangle order; isosurface_kernels.cuh) from only the blocks of kIsoBlock³ cells whose certified
// bounds (bounds_kernels.cuh) reach iso. DESIGN §15 has the argument why the skipped blocks hold no crossing edge.
//
// Block (bi, bj, bk) owns the cells [16 b, min(16 b + 16, n)) per axis and the points of the same half-open range, plus the
// points of index n on every axis where it is the last block. Its key is bi | bj << 10 | bk << 20, so ascending keys are
// block-linear order. A block's (B+1)³ values cover every edge its points own and every corner of its cells.
//   isoCullBoxesKernel    the closed boxes [P(c0), P(min(c0 + s, n))] of blocks of s cells (isoCoord, so monotone in c)
//   isoCullSplitKernel    uncertified blocks: their children of s/2 cells, or at the leaf level the block itself
//   isoRowWeightsKernel   rows per block (owned point / cell rows along y, and y times z), scanned for the row ranks
//   isoRowMetaKernel      per block the rank of its local row (lj, lk) among all rows of the grid in the dense order
//   isoBlockCountKernel   per block the values, per owned point mask | earlier vertices of its row << 8, per row the counts
//   isoBlockEmitKernel    per block the values again, its vertices, and the triangles of its cells
#pragma once
#include "isosurface_kernels.cuh"

namespace hpsdf
{
    constexpr uint32_t kIsoBlockSmem = 4096 * 4 + kIsoBlockPts * 8;        // top table + the block's values

    __device__ __forceinline__ uint32_t isoKey(uint32_t i, uint32_t j, uint32_t k) { return i | (j << 10) | (k << 20); }

    __global__ void isoCullTopKernel(const uint32_t nx, const uint32_t ny, const uint32_t n, uint32_t* __restrict__ keys)
    {
        const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
        if (t < n) keys[t] = isoKey(t % nx, (t / nx) % ny, t / (nx * ny));
    }

    __global__ void isoCullBoxesKernel(const IsoGrid g, const uint32_t s, const uint32_t* __restrict__ keys, uint32_t m,
                                       double* __restrict__ lo, double* __restrict__ hi)
    {
        const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
        if (t >= m) return;
        const uint32_t key = keys[t];
        #pragma unroll
        for (int a = 0; a < 3; ++a)
        {
            const uint32_t c0 = ((key >> (10 * a)) & 1023u) * s, c1 = min(c0 + s, g.n[a]);
            lo[3 * t + a] = isoCoord(g, a, c0);
            hi[3 * t + a] = isoCoord(g, a, c1);
        }
    }

    // Certified: f_lo >= iso (every point outside) or f_hi < iso (every point inside). NaN bounds certify nothing; iso = NaN
    // certifies everything, since no point has V < NaN, so no edge crosses. counters[0] = uncertified blocks, [1] = keys written.
    __global__ void isoCullSplitKernel(const IsoGrid g, const uint32_t childCells, const uint32_t* __restrict__ keys, uint32_t m,
                                       const double* __restrict__ fLo, const double* __restrict__ fHi, uint32_t* __restrict__ out,
                                       uint32_t* __restrict__ counters)
    {
        const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
        if (t >= m || g.iso != g.iso || fLo[t] >= g.iso || fHi[t] < g.iso) return;
        atomicAdd(counters, 1u);
        const uint32_t key = keys[t];
        if (!childCells) { out[atomicAdd(counters + 1, 1u)] = key; return; }
        const uint32_t b[3] = { key & 1023u, (key >> 10) & 1023u, key >> 20 };
        for (int c = 0; c < 8; ++c)
        {
            uint32_t ch[3];
            bool in = true;
            #pragma unroll
            for (int a = 0; a < 3; ++a) { ch[a] = 2 * b[a] + ((c >> a) & 1); in = in && ch[a] * childCells < g.n[a]; }
            if (in) out[atomicAdd(counters + 1, 1u)] = isoKey(ch[0], ch[1], ch[2]);
        }
    }

    // The shape of one leaf block: origin cell o, cells e per axis (the block's points are o .. o + e), owned points op.
    struct IsoBlockShape { uint32_t o[3], e[3], op[3]; };

    __device__ __forceinline__ IsoBlockShape isoShape(const IsoGrid& g, uint32_t key)
    {
        IsoBlockShape s;
        #pragma unroll
        for (int a = 0; a < 3; ++a)
        {
            s.o[a] = ((key >> (10 * a)) & 1023u) * kIsoBlock;
            s.e[a] = min(kIsoBlock, g.n[a] - s.o[a]);
            s.op[a] = s.o[a] + kIsoBlock >= g.n[a] ? s.e[a] + 1 : kIsoBlock;      // the last block also owns point n
        }
        return s;
    }

    __device__ __forceinline__ uint32_t isoLowerBound(const uint32_t* __restrict__ keys, uint32_t n, uint32_t key)
    {
        uint32_t lo = 0, hi = n;
        while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (keys[mid] < key) lo = mid + 1; else hi = mid; }
        return lo;
    }

    // w[0..3][b]: owned point rows along y, point rows of the block (y times z), the same for cell rows; w[.][n] = 0
    __global__ void isoRowWeightsKernel(const IsoGrid g, const uint32_t* __restrict__ keys, uint32_t n, unsigned long long* __restrict__ w)
    {
        const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
        if (b > n) return;
        const size_t stride = (size_t)n + 1;
        unsigned long long r[4] = { 0, 0, 0, 0 };
        if (b < n)
        {
            const IsoBlockShape s = isoShape(g, keys[b]);
            r[0] = s.op[1]; r[1] = (unsigned long long)s.op[1] * s.op[2];
            r[2] = s.e[1];  r[3] = (unsigned long long)s.e[1] * s.e[2];
        }
        for (int k = 0; k < 4; ++k) w[k * stride + b] = r[k];
    }

    // Rows in the dense order: slab bk, then local row lk, then block row group (bk, bj) ascending bj, then local row lj, then
    // the group's blocks in ascending bi. With ps the exclusive scans of isoRowWeightsKernel over the sorted blocks, slab
    // [s0, s1) and group [g0, g1): rank(b, lj, lk) = ps_yz[s0] + lk (ps_y[s1] - ps_y[s0]) + (ps_y[g0] - ps_y[s0]) + lj (g1 - g0) + b - g0.
    __global__ void isoRowMetaKernel(const uint32_t* __restrict__ keys, uint32_t n, const unsigned long long* __restrict__ ps,
                                     IsoRowMeta* __restrict__ metaV, IsoRowMeta* __restrict__ metaT)
    {
        const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
        if (b >= n) return;
        const uint32_t key = keys[b], slab = key & ~((1u << 20) - 1), grp = key & ~1023u;
        const uint32_t s0 = isoLowerBound(keys, n, slab), s1 = isoLowerBound(keys, n, slab + (1u << 20));
        const uint32_t g0 = isoLowerBound(keys, n, grp), g1 = isoLowerBound(keys, n, grp + 1024u);
        const size_t stride = (size_t)n + 1;
        for (int k = 0; k < 2; ++k)
        {
            const unsigned long long* py = ps + 2 * k * stride, *pyz = py + stride;
            IsoRowMeta mt;
            mt.strideK = py[s1] - py[s0];
            mt.strideJ = g1 - g0;
            mt.base = pyz[s0] + (py[g0] - py[s0]) + (b - g0);
            (k ? metaT : metaV)[b] = mt;
        }
    }

    __device__ __forceinline__ unsigned long long isoRank(const IsoRowMeta& m, uint32_t lj, uint32_t lk)
    {
        return m.base + lk * m.strideK + lj * m.strideJ;
    }

    // The block's values at local points li + 17 (lj + 17 lk), li <= e[0] etc., with isoGridKernel's evaluation: a warp takes
    // 32 consecutive local points, findLeaf + evalWarp, so every value is hpsdf_query's bit for bit.
    __device__ __forceinline__ void isoBlockValues(const DeviceTreeView& view, const uint32_t* top, const IsoGrid& g, const IsoBlockShape& s,
                                                   double* __restrict__ sV)
    {
        const uint32_t lane = threadIdx.x & 31;
        for (uint32_t base = threadIdx.x & ~31u; base < kIsoBlockPts; base += blockDim.x)
        {
            const uint32_t p = base + lane, li = p % kIsoSide, r = p / kIsoSide, lj = r % kIsoSide, lk = r / kIsoSide;
            const bool valid = p < kIsoBlockPts && li <= s.e[0] && lj <= s.e[1] && lk <= s.e[2];
            LeafHit h;
            if (valid) h = findLeaf(view, top, isoCoord(g, 0, s.o[0] + li), isoCoord(g, 1, s.o[1] + lj), isoCoord(g, 2, s.o[2] + lk));
            const double v = evalWarp(h, view.bidx);
            if (valid) sV[p] = v;
        }
    }

    __device__ __forceinline__ uint32_t isoCellLabel(const double* __restrict__ sV, uint32_t p, double iso)
    {
        uint32_t lab = 0;
        #pragma unroll
        for (int c = 0; c < 8; ++c)
            if (sV[p + (c & 1) + ((c & 2) ? kIsoSide : 0u) + ((c & 4) ? kIsoSide * kIsoSide : 0u)] < iso) lab |= 1u << c;
        return lab;
    }

    // One CTA per active block; one thread per owned row of points, then per row of cells.
    __global__ void __launch_bounds__(kQueryThreads, kQueryBlocksPerSm)
    isoBlockCountKernel(const DeviceTreeView view, const IsoGrid g, const IsoBlocks B)
    {
        extern __shared__ __align__(16) unsigned char sDyn[];
        uint32_t (&sTop)[4096] = *reinterpret_cast<uint32_t(*)[4096]>(sDyn);
        double* sV = reinterpret_cast<double*>(sDyn + 4096 * 4);
        const bool useTop = stageTop(sTop, view.top);
        const uint32_t b = blockIdx.x;
        const IsoBlockShape s = isoShape(g, B.keys[b]);
        isoBlockValues(view, useTop ? sTop : nullptr, g, s, sV);
        __syncthreads();
        const IsoRowMeta mv = B.metaV[b], mt = B.metaT[b];
        uint16_t* tab = B.tab + (size_t)b * kIsoBlockPts;
        for (uint32_t r = threadIdx.x; r < s.op[1] * s.op[2]; r += blockDim.x)
        {
            const uint32_t lj = r % s.op[1], lk = r / s.op[1];
            uint32_t run = 0;
            for (uint32_t li = 0; li < s.op[0]; ++li)
            {
                const uint32_t p = li + kIsoSide * (lj + kIsoSide * lk);
                const bool in0 = sV[p] < g.iso;
                uint32_t m = 0;
                #pragma unroll
                for (int d = 1; d < 8; ++d)
                {
                    const uint32_t dx = d & 1, dy = (d >> 1) & 1, dz = d >> 2;
                    if (li + dx > s.e[0] || lj + dy > s.e[1] || lk + dz > s.e[2]) continue;
                    if ((sV[p + dx + kIsoSide * (dy + kIsoSide * dz)] < g.iso) != in0) m |= 1u << (d - 1);
                }
                tab[p] = (uint16_t)(m | (run << 8));
                run += __popc(m);
            }
            B.cntV[isoRank(mv, lj, lk)] = run;
        }
        for (uint32_t r = threadIdx.x; r < s.e[1] * s.e[2]; r += blockDim.x)
        {
            const uint32_t lj = r % s.e[1], lk = r / s.e[1];
            uint32_t run = 0;
            for (uint32_t li = 0; li < s.e[0]; ++li) run += c_isoCellTris[isoCellLabel(sV, li + kIsoSide * (lj + kIsoSide * lk), g.iso)];
            B.cntT[isoRank(mt, lj, lk)] = run;
        }
    }

    // Vertices and triangles of one active block with isoEmitKernel's and isoTriKernel's arithmetic and order. A triangle edge
    // owned by a point past the block's owned range is owned by the +x / +y / +z neighbour (or a diagonal one), which is active.
    __global__ void __launch_bounds__(kQueryThreads, kQueryBlocksPerSm)
    isoBlockEmitKernel(const DeviceTreeView view, const IsoGrid g, const IsoBlocks B, float* __restrict__ verts, uint32_t* __restrict__ tris)
    {
        extern __shared__ __align__(16) unsigned char sDyn[];
        __shared__ uint32_t sNbr[8];
        uint32_t (&sTop)[4096] = *reinterpret_cast<uint32_t(*)[4096]>(sDyn);
        double* sV = reinterpret_cast<double*>(sDyn + 4096 * 4);
        const uint32_t b = blockIdx.x, key = B.keys[b];
        if (threadIdx.x < 8)
        {
            const uint32_t sh = threadIdx.x;
            const uint32_t k = isoKey((key & 1023u) + (sh & 1), ((key >> 10) & 1023u) + ((sh >> 1) & 1), (key >> 20) + (sh >> 2));
            const uint32_t at = sh ? isoLowerBound(B.keys, B.n, k) : b;
            sNbr[sh] = at < B.n && B.keys[at] == k ? at : 0xFFFFFFFFu;
        }
        const bool useTop = stageTop(sTop, view.top);
        const IsoBlockShape s = isoShape(g, key);
        isoBlockValues(view, useTop ? sTop : nullptr, g, s, sV);
        __syncthreads();
        const uint16_t* tab = B.tab + (size_t)b * kIsoBlockPts;
        const IsoRowMeta mv = B.metaV[b], mt = B.metaT[b];
        for (uint32_t r = threadIdx.x; r < s.op[1] * s.op[2]; r += blockDim.x)
        {
            const uint32_t lj = r % s.op[1], lk = r / s.op[1];
            unsigned long long o = B.baseV[isoRank(mv, lj, lk)];
            for (uint32_t li = 0; li < s.op[0]; ++li)
            {
                const uint32_t p = li + kIsoSide * (lj + kIsoSide * lk), m = tab[p] & 0x7Fu;
                if (!m) continue;
                const uint32_t idx[3] = { s.o[0] + li, s.o[1] + lj, s.o[2] + lk };
                const double v0 = sV[p];
                const double x0[3] = { isoCoord(g, 0, idx[0]), isoCoord(g, 1, idx[1]), isoCoord(g, 2, idx[2]) };
                for (int d = 1; d < 8; ++d)
                {
                    if (!((m >> (d - 1)) & 1)) continue;
                    const uint32_t q = p + (d & 1) + ((d & 2) ? kIsoSide : 0u) + ((d & 4) ? kIsoSide * kIsoSide : 0u);
                    const double t = __ddiv_rn(__dsub_rn(g.iso, v0), __dsub_rn(sV[q], v0));
                    #pragma unroll
                    for (int a = 0; a < 3; ++a)
                    {
                        const double x1 = ((d >> a) & 1) ? isoCoord(g, a, idx[a] + 1) : x0[a];
                        verts[3 * o + a] = __double2float_rn(__dadd_rn(x0[a], __dmul_rn(t, __dsub_rn(x1, x0[a]))));
                    }
                    ++o;
                }
            }
        }
        for (uint32_t r = threadIdx.x; r < s.e[1] * s.e[2]; r += blockDim.x)
        {
            const uint32_t lj = r % s.e[1], lk = r / s.e[1];
            unsigned long long o = B.baseT[isoRank(mt, lj, lk)];
            for (uint32_t li = 0; li < s.e[0]; ++li)
            {
                const uint32_t lab = isoCellLabel(sV, li + kIsoSide * (lj + kIsoSide * lk), g.iso);
                if (lab == 0 || lab == 0xFF) continue;
                for (int t = 0; t < 6; ++t)
                {
                    uint32_t L = 0;
                    #pragma unroll
                    for (int c = 0; c < 4; ++c) L |= ((lab >> c_isoChain[t][c]) & 1u) << c;
                    const IsoTetCase cs = c_isoTet[t][L];
                    for (int e = 0; e < 3 * cs.n; ++e)
                    {
                        const uint32_t off = cs.e[e] & 7, d = cs.e[e] >> 3;
                        uint32_t q[3] = { li + (off & 1), lj + ((off >> 1) & 1), lk + (off >> 2) }, sh = 0;
                        #pragma unroll
                        for (int a = 0; a < 3; ++a)
                            if (q[a] >= s.op[a]) { sh |= 1u << a; q[a] -= kIsoBlock; }
                        const uint32_t nb = sNbr[sh];
                        uint32_t vi = 0xFFFFFFFFu;                  // a missing neighbour would break the culling argument
                        if (nb != 0xFFFFFFFFu)
                        {
                            const uint32_t ent = B.tab[(size_t)nb * kIsoBlockPts + q[0] + kIsoSide * (q[1] + kIsoSide * q[2])];
                            vi = (uint32_t)(B.baseV[isoRank(B.metaV[nb], q[1], q[2])] + (ent >> 8) + __popc(ent & ((1u << (d - 1)) - 1u)));
                        }
                        tris[3 * o + e] = vi;
                    }
                    o += cs.n;
                }
            }
        }
    }
}
