// query_kernels.cuh — batched Octree::Query (Source/HP/Octree.cpp:662-702): the reference has no batch API
// (callers loop over Query, HPBenchmarks.cpp:107-110); this is the data-parallel form.
//
// Layout: points are AoS n x 3 f64 (the Eigen::Vector3d array a caller already has). A CTA stages a tile of 256 points
// (6 KB) into shared memory with coalesced 16-byte loads, then each thread evaluates one point. The 4096-entry top-of-tree
// table (16 KB) is staged once per CTA; the grid is persistent (a few CTAs per SM looping over tiles) so that staging
// amortises. Algorithmic HBM traffic: 24 B in + 8 B out per point; the tree (16 B nodes + padded coefficients) stays in L2.
#pragma once
#include "query_eval.cuh"

namespace hpsdf
{
    constexpr int kQueryThreads = 256;
#ifndef HPSDF_QUERY_MINBLOCKS
#define HPSDF_QUERY_MINBLOCKS 4
#endif
    constexpr int kQueryBlocksPerSm = HPSDF_QUERY_MINBLOCKS;

    // Stage the 4096-entry top table of the tree into shared memory once per CTA of a persistent kernel (all threads must
    // call this); false when the tree has none. The only block-wide barrier: the table is read-only afterwards. Callers
    // pick sTop or nullptr where they descend: a returned table pointer stays live across their loops and made queryKernel
    // and isoGridKernel spill more.
    __device__ __forceinline__ bool stageTop(uint32_t (&sTop)[4096], const uint32_t* top)
    {
        if (!top) return false;
        for (int i = threadIdx.x; i < 1024; i += kQueryThreads)
            reinterpret_cast<uint4*>(sTop)[i] = __ldg(reinterpret_cast<const uint4*>(top) + i);
        __syncthreads();
        return true;
    }

    __global__ void __launch_bounds__(kQueryThreads, kQueryBlocksPerSm)
    queryKernel(const DeviceTreeView view, const double* __restrict__ xyz, size_t n, double* __restrict__ out,
                const int aligned /* xyz starts on a 16-byte boundary */)
    {
        __shared__ uint32_t sTop[4096];
        __shared__ __align__(16) double sPts[kQueryThreads / 32][96];          // per warp: 32 points x 3 doubles
        const bool useTop = stageTop(sTop, view.top);
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const size_t nGroups = (n + 31) / 32;                                   // a warp handles 32 consecutive points
        const size_t warpsTotal = (size_t)gridDim.x * (kQueryThreads / 32);
        double* sp = sPts[warp];
        for (size_t g = (size_t)blockIdx.x * (kQueryThreads / 32) + warp; g < nGroups; g += warpsTotal)
        {
            const size_t base = g * 32;
            const size_t cnt = n - base < 32 ? n - base : 32;
            const double* src = xyz + 3 * base;                                 // 32 * 24 B = 768 B: 16-byte aligned
            if (cnt == 32 && aligned)
            {
                reinterpret_cast<double2*>(sp)[lane] = __ldcs(reinterpret_cast<const double2*>(src) + lane);
                if (lane < 16) reinterpret_cast<double2*>(sp)[32 + lane] = __ldcs(reinterpret_cast<const double2*>(src) + 32 + lane);
            }
            else
                for (size_t v = lane; v < 3 * cnt; v += 32) sp[v] = src[v];
            __syncwarp();
            LeafHit h;
            if ((size_t)lane < cnt) h = findLeaf(view, useTop ? sTop : nullptr, sp[3 * lane], sp[3 * lane + 1], sp[3 * lane + 2]);
            __syncwarp();                           // sp is overwritten by the next group
            const double v = evalWarp(h, view.bidx);
            if ((size_t)lane < cnt) __stcs(out + base + lane, v);
        }
    }

#ifndef HPSDF_DERIV1_MINBLOCKS
#define HPSDF_DERIV1_MINBLOCKS 3
#endif
#ifndef HPSDF_DERIV2_MINBLOCKS
#define HPSDF_DERIV2_MINBLOCKS 2
#endif
    // CTAs per SM of queryDerivativesKernel<ORDER>: they set its register budget (DESIGN.md §13 has the ptxas lines)
    constexpr int derivBlocksPerSm(int order) { return order == 1 ? HPSDF_DERIV1_MINBLOCKS : HPSDF_DERIV2_MINBLOCKS; }

    // hpsdf_query_derivatives (DESIGN.md §13): Query's value and the exact gradient (ORDER 1) and Hessian (ORDER 2) of the
    // hit leaf's polynomial in user space, d/dx_a = s_a d/du_a with s_a = 2^(depth+1) invSizes_a; 0 outside the root.
    // queryKernel's structure: persistent grid, warp tiles of 32 points staged through shared memory, the top table in
    // shared memory, warp-uniform degree dispatch. The value is evalLeafMasked's / evalLeafGeneric's, so Query's to the bit.
    // The tile buffer also stages the gradients and Hessians, so every store of a warp is one contiguous run.
    template <int ORDER>
    __global__ void __launch_bounds__(kQueryThreads, derivBlocksPerSm(ORDER))
    queryDerivativesKernel(const DeviceTreeView view, const double* __restrict__ xyz, size_t n, double* __restrict__ value,
                           double* __restrict__ grad, double* __restrict__ hess, const int aligned /* xyz is 16-byte aligned */)
    {
        constexpr int kTile = ORDER == 2 ? 6 * 32 : 3 * 32;
        __shared__ uint32_t sTop[4096];
        __shared__ __align__(16) double sBuf[kQueryThreads / 32][kTile];
        const bool useTop = stageTop(sTop, view.top);
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const size_t nGroups = (n + 31) / 32;
        const size_t warpsTotal = (size_t)gridDim.x * (kQueryThreads / 32);
        double* sp = sBuf[warp];
        for (size_t g = (size_t)blockIdx.x * (kQueryThreads / 32) + warp; g < nGroups; g += warpsTotal)
        {
            const size_t base = g * 32;
            const size_t cnt = n - base < 32 ? n - base : 32;
            const double* src = xyz + 3 * base;
            if (cnt == 32 && aligned)
            {
                reinterpret_cast<double2*>(sp)[lane] = __ldcs(reinterpret_cast<const double2*>(src) + lane);
                if (lane < 16) reinterpret_cast<double2*>(sp)[32 + lane] = __ldcs(reinterpret_cast<const double2*>(src) + 32 + lane);
            }
            else
                for (size_t v = lane; v < 3 * cnt; v += 32) sp[v] = src[v];
            __syncwarp();
            LeafHit h;
            if ((size_t)lane < cnt) h = findLeaf(view, useTop ? sTop : nullptr, sp[3 * lane], sp[3 * lane + 1], sp[3 * lane + 2]);
            __syncwarp();                           // sp now takes this tile's results
            LeafDerivs d;
            double v;
            switch ((int)__reduce_max_sync(0xFFFFFFFFu, (unsigned)(h.degree < 0 ? 0 : h.degree)))
            {
                case 0:  v = evalLeafMasked<0, ORDER>(h.coeffs, h.degree, h.ux, h.uy, h.uz, h.depth, &d); break;
                case 1:  v = evalLeafMasked<1, ORDER>(h.coeffs, h.degree, h.ux, h.uy, h.uz, h.depth, &d); break;
                case 2:  v = evalLeafMasked<2, ORDER>(h.coeffs, h.degree, h.ux, h.uy, h.uz, h.depth, &d); break;
                case 3:  v = evalLeafMasked<3, ORDER>(h.coeffs, h.degree, h.ux, h.uy, h.uz, h.depth, &d); break;
                case 4:  v = evalLeafMasked<4, ORDER>(h.coeffs, h.degree, h.ux, h.uy, h.uz, h.depth, &d); break;
                case 5:  v = evalLeafMasked<5, ORDER>(h.coeffs, h.degree, h.ux, h.uy, h.uz, h.depth, &d); break;
                case 6:  v = evalLeafMasked<6, ORDER>(h.coeffs, h.degree, h.ux, h.uy, h.uz, h.depth, &d); break;
                default:
                    v = 0.0;
                    if (h.degree >= 0)
                    {
                        v = evalLeafGeneric(h.coeffs, h.degree, h.ux, h.uy, h.uz, h.depth, view.bidx);
                        const double u[3] = { h.ux, h.uy, h.uz };
                        leafDerivsGeneric<ORDER>(h.coeffs, h.degree, h.depth, u, view.bidx, d);
                    }
                    break;
            }
            const double scale = (double)(2u << h.depth);
            const double s[3] = { scale * view.map.invSizes[0], scale * view.map.invSizes[1], scale * view.map.invSizes[2] };
            const bool in = h.degree >= 0;                                          // outside the root: DBL_MAX, derivatives 0
            if ((size_t)lane < cnt) __stcs(value + base + lane, in ? v : DBL_MAX);
            #pragma unroll
            for (int a = 0; a < 3; ++a) sp[3 * lane + a] = in ? d.g[a] * s[a] : 0.0;
            __syncwarp();
            for (size_t k = lane; k < 3 * cnt; k += 32) __stcs(grad + 3 * base + k, sp[k]);
            if constexpr (ORDER == 2)
            {
                __syncwarp();
                constexpr int ia[6] = { 0, 0, 0, 1, 1, 2 }, ib[6] = { 0, 1, 2, 1, 2, 2 };
                #pragma unroll
                for (int k = 0; k < 6; ++k) sp[6 * lane + k] = in ? d.h[k] * (s[ia[k]] * s[ib[k]]) : 0.0;
                __syncwarp();
                for (size_t k = lane; k < 6 * cnt; k += 32) __stcs(hess + 6 * base + k, sp[k]);
            }
            __syncwarp();                           // sp is overwritten by the next tile
        }
    }

    // Octree::QueryWithGradient (Octree.cpp:749-789) / FApproxWithGradient (:904-985): central differences with eps = 1e-4
    // in the leaf's local coordinate, gradient normalised. One thread per point, generic-degree loops (not a hot path).
    __global__ void __launch_bounds__(256)
    queryGradientKernel(const DeviceTreeView view, const double* __restrict__ xyz, size_t n, double* __restrict__ out,
                        double* __restrict__ grad)
    {
        const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (t >= n) return;
        const LeafHit h = findLeaf(view, view.top, xyz[3 * t], xyz[3 * t + 1], xyz[3 * t + 2]);
        if (h.degree < 0) { out[t] = DBL_MAX; return; }
        const int depth = h.depth, degree = h.degree;
        const double* coeffs = h.coeffs;
        const uint32_t* bidx = view.bidx;
        const double eps = 0.0001, u[3] = { h.ux, h.uy, h.uz };
        double lut[kMaxDegree + 1][3][3];
        for (int a = 0; a < 3; ++a)
        {
            const double us[3] = { u[a], u[a] + eps, u[a] - eps };
            for (int v = 0; v < 3; ++v)
            {
                lut[0][a][v] = c_nl[0][depth];
                double m2 = 0.0, m1 = 1.0, l = 1.0;
                for (int j = 1; j <= degree; ++j)
                {
                    l = c_rec[j][0] * us[v] * m1 - c_rec[j][1] * m2; m2 = m1; m1 = l;
                    lut[j][a][v] = l * c_nl[j][depth];
                }
            }
        }
        const int nc = coeffCount(degree);
        double g[3];
        for (int k = 0; k < 3; ++k)
        {
            double fp = 0.0, fm = 0.0;
            for (int i = 0; i < nc; ++i)
            {
                const int a = (bidx[i] >> (8 * k)) & 0xFF;
                fp += coeffs[i] * lut[a][k][1]; fm += coeffs[i] * lut[a][k][2];            // Octree.cpp:961-965
            }
            g[k] = (fp - fm) / (2.0 * eps);
        }
        const double nrm = sqrt(g[0] * g[0] + (g[1] * g[1] + g[2] * g[2]));
        if (nrm > 0.0) { g[0] /= nrm; g[1] /= nrm; g[2] /= nrm; }
        double f = 0.0;
        for (int i = 0; i < nc; ++i)
        {
            const uint32_t abc = bidx[i];
            f += coeffs[i] * ((lut[abc & 0xFF][0][0] * lut[(abc >> 8) & 0xFF][1][0]) * lut[(abc >> 16) & 0xFF][2][0]);
        }
        out[t] = f;
        grad[3 * t] = g[0]; grad[3 * t + 1] = g[1]; grad[3 * t + 2] = g[2];
    }

    __global__ void gatherSegmentsKernel(const double* __restrict__ src, double* __restrict__ dst, const uint32_t* __restrict__ srcOff,
                                         const uint32_t* __restrict__ dstOff, const uint32_t* __restrict__ count, uint32_t nSeg)
    {
        // one warp per segment
        const uint32_t seg = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
        if (seg >= nSeg) return;
        const double* s = src + srcOff[seg];
        double* d = dst + dstOff[seg];
        for (uint32_t i = lane; i < count[seg]; i += 32) d[i] = s[i];
    }

    // Octree::QueryRay (Source/HP/Octree.cpp:705-746) + Ray::Ray / Ray::IntersectAABB (Source/HP/Ray.cpp:5-65), one ray per
    // thread, statement by statement — including what the reference does with its own intermediate results: the origin is
    // moved into the unit cube but the direction is not rescaled (:713); when the origin is outside the root, the vector the
    // march starts from is the `a_` output of IntersectAABB, whose x component holds the entry PARAMETER and whose y, z
    // components hold the slab parameters of those axes (:715-719, Ray.cpp:27-61), not a point; every sample goes through
    // Query, which applies the root map a second time (:729, :665); `t_` receives the last field value, not a distance
    // (:733). For the default root box and origins inside it these coincide with sphere tracing of the field.
    __global__ void __launch_bounds__(256)
    queryRayKernel(const DeviceTreeView view, const double* __restrict__ origins, const double* __restrict__ dirs, size_t n,
                   const double tMax, unsigned char* __restrict__ hit, double* __restrict__ tOut)
    {
        const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n) return;
        constexpr unsigned MAX_STEPS = 200;
        constexpr double eps = 0.0001, minStep = 0.0001;
        const RootMap& map = view.map;
        double o[3], dir[3], inv[3];
        int sign[3];
        for (int a = 0; a < 3; ++a)
        {
            o[a] = (origins[3 * i + a] - map.centre[a]) * map.invSizes[a];                     // :713
            dir[a] = dirs[3 * i + a];
            inv[a] = 1.0 / dir[a];                                                              // Ray.cpp:10
            sign[a] = inv[a] < 0.0;                                                             // Ray.cpp:11-13
        }
        double intMin[3] = { o[0], o[1], o[2] };
        const float fx = (float)o[0], fy = (float)o[1], fz = (float)o[2];
        const bool inside = fx >= -0.5f && fx <= 0.5f && fy >= -0.5f && fy <= 0.5f && fz >= -0.5f && fz <= 0.5f;      // nodes[0].aabb.contains
        bool ok = true;
        if (!inside)
        {
            const double bounds[2] = { -0.5, 0.5 };
            double a_[3] = { o[0], o[1], o[2] }, b_[3] = { 0.0, 0.0, 0.0 };
            a_[0] = (bounds[sign[0]] - o[0]) * inv[0];     b_[0] = (bounds[1 - sign[0]] - o[0]) * inv[0];     // Ray.cpp:27-30
            a_[1] = (bounds[sign[1]] - o[1]) * inv[1];     b_[1] = (bounds[1 - sign[1]] - o[1]) * inv[1];
            if ((a_[0] > b_[1]) || (a_[1] > b_[0])) ok = false;                                                // :32-35
            if (ok)
            {
                if (a_[1] > a_[0]) a_[0] = a_[1];                                                              // :37-40
                if (b_[1] < b_[0]) b_[0] = b_[1];                                                              // :42-45
                a_[2] = (bounds[sign[2]] - o[2]) * inv[2]; b_[2] = (bounds[1 - sign[2]] - o[2]) * inv[2];     // :47-48
                if ((a_[0] > b_[2]) || (a_[2] > b_[0])) ok = false;                                            // :50-53
                if (ok)
                {
                    if (a_[2] > a_[0]) a_[0] = a_[2];                                                          // :55-58
                    intMin[0] = a_[0]; intMin[1] = a_[1]; intMin[2] = a_[2];
                }
            }
        }
        unsigned char h = 0;
        double t = 0.0;
        if (ok)
        {
            double d = 0.0;
            for (unsigned s = 0; s < MAX_STEPS; ++s)
            {
                const double v = treeQuery(view, intMin[0] + d * dir[0], intMin[1] + d * dir[1], intMin[2] + d * dir[2]);
                if (v < eps) { t = v; h = 1; break; }                                           // :731-736
                d += v * 0.95 + minStep;                                                        // :739
                if (d > tMax) break;                                                            // :741-744
            }
        }
        hit[i] = h;
        tOut[i] = t;
    }
}
