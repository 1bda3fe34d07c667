// bounds_kernels.cuh — hpsdf_query_bounds: certified bounds of the field over axis-aligned boxes (DESIGN §14).
//
// A box maps to [P_lo, P_hi] in the unit cube with Query's root map. Query keeps a point whose f32 cast lies in
// [-0.5, 0.5], which in f64 is |p| <= L = 0.5 + 2^-25; a node's extended cell E(node) is its closed cell, widened to L on
// faces on the root's boundary. Each leaf whose E(leaf) meets the box contributes an interval: the hull of the degree-(p,p,p)
// tensor Bernstein coefficients of its polynomial on the box clipped to E(leaf), widened by A_leaf = kappa_p 2^-53 S_leaf
// (S_leaf = sum |c_i| nl[a_i] nl[b_i] nl[c_i]), intersected with the leaf's interval over all of E(leaf). The result is the
// min and max over those intervals, and DBL_MAX as the upper bound when part of the box is outside the root.
//
// Per axis the Bernstein form of every normalised Legendre polynomial N_j on the sub-interval [ua, ub] is
// M[j][k] = sum_i Binv[k][i] N_j(u_i), with u_i the Chebyshev-Lobatto nodes of [ua, ub] and Binv the inverse collocation
// matrix raycast uses (c_rayNodes, c_rayBern). The tensor coefficients B[k1][k2][k3] = sum c (Mx My Mz) are contracted by sum
// factorisation: z, then y, then x, with a running min and max; the (p+1)^3 tensor is never stored.
//
// A per-node table of enclosures (16 B per node) is built on a tree's first bounds query: a leaf's entry is its interval over
// E(leaf), an internal node's the min and max of its children's. boundsKernel walks a warp-wide stack from the root: a node
// that misses the box is dropped, one whose entry lies inside the running interval cannot change the result and is dropped,
// one the box covers contributes its entry, and the rest push their children or, for leaves, run the sub-box hull. Min and
// max are exact, a covered node's entry is what its descent would give, and a leaf's sub-box interval lies inside its entry,
// so the result does not depend on the order of the walk or on pruning.
#pragma once
#include "raycast_kernels.cuh"

namespace hpsdf
{
    // Containment bound of Query in f64: |p| <= 0.5 + 2^-25 casts to an f32 in [-0.5, 0.5] (the tie rounds to even, 0.5).
    constexpr double kBoundsL = 0.5 + 0x1p-25;
    // log2 of kappa_p, the rounding allowance per degree in units of 2^-53 S_leaf: DESIGN §14 derives
    // G^3 (Q_p + 3 W_p E_p + (3p + 4) W_p) and rounds it up to a power of two.
    constexpr int kBoundsKappaLog2[kMaxDegree + 1] = { 5, 7, 11, 13, 16, 18, 21, 23, 26, 28, 30, 32, 35 };
    constexpr int kBoundsThreads = 64;          // two warps per CTA: 2 x 20 KB of stack
    // Stack entries per warp. Each round pops the top min(32, size) entries and pushes at most 8 children per entry. The
    // remnants of push batches on the stack have strictly increasing smallest depths from bottom to top (children are one
    // level below the shallowest entry popped), and depths 1..10 hold such batches of at most 256 entries: 2560.
    constexpr int kBoundsStack = 10 * 256;

    // Closed extended cell [lo, hi] of the cell i (0 <= i < 2^d) of depth d along one axis, and its centre.
    __device__ __forceinline__ void boundsCell(int d, uint32_t i, double& lo, double& hi, double& c)
    {
        const double size = ldexp(1.0, -d);
        const double a = (double)i * size - 0.5;
        c = a + 0.5 * size;
        lo = i == 0 ? -kBoundsL : a;
        hi = i + 1 == (1u << d) ? kBoundsL : a + size;
    }

    // Interval of a degree-P leaf polynomial over the box u in [ua, ub] (per axis, in the leaf's local coordinates): the hull of
    // its tensor Bernstein coefficients widened by A_leaf. Out of line: one call per hull is nothing against its O(p^4) FMAs,
    // and its arrays stay out of the register budget of the callers.
    template <int P>
    __device__ __noinline__ double2 leafHull(const double* __restrict__ coeffs, int depth, const double (&ua)[3], const double (&ub)[3])
    {
        constexpr int N = P + 1, NC = coeffCount(P);
        double M[3][N][N];                                  // M[axis][j][k]: Bernstein coefficient k of N_j on [ua, ub]
        #pragma unroll 1
        for (int a = 0; a < 3; ++a)
        {
            double nv[N][N];                                // nv[i][j] = N_j(u_i)
            #pragma unroll
            for (int i = 0; i <= P; ++i)
            {
                const double u = i == 0 ? ua[a] : i == P ? ub[a] : fma(c_rayNodes[rayNodeOffset(P) + i], ub[a] - ua[a], ua[a]);
                nv[i][0] = c_nl[0][depth];
                double m2 = 0.0, m1 = 1.0;
                #pragma unroll
                for (int j = 1; j <= P; ++j)
                {
                    const double v = c_rec[j][0] * u * m1 - c_rec[j][1] * m2; m2 = m1; m1 = v;
                    nv[i][j] = v * c_nl[j][depth];
                }
            }
            #pragma unroll
            for (int j = 0; j <= P; ++j)
                #pragma unroll
                for (int k = 0; k <= P; ++k)
                {
                    double s = 0.0;
                    #pragma unroll
                    for (int i = 0; i <= P; ++i) s = fma(c_rayBern[rayBernOffset(P) + k * N + i], nv[i][j], s);
                    M[a][j][k] = s;
                }
        }
        // S_leaf, rounded up
        double sAbs = 0.0;
        {
            int idx = 0;
            #pragma unroll
            for (int p = 0; p <= P; ++p)
                #pragma unroll
                for (int i = 0; i <= p; ++i)
                    #pragma unroll
                    for (int j = 0; j <= p - i; ++j, ++idx)
                        if (idx < NC)
                            sAbs = __fma_ru(fabs(__ldg(coeffs + idx)), __dmul_ru(__dmul_ru(c_nl[i][depth], c_nl[j][depth]), c_nl[p - i - j][depth]), sAbs);
        }
        double mn = __longlong_as_double(0x7FF0000000000000ll), mx = -mn;
        #pragma unroll 1
        for (int k3 = 0; k3 <= P; ++k3)
        {
            double S[N][N];                                 // S[a][b] = sum_c coef(a, b, c) Mz[c][k3], a + b <= P
            #pragma unroll
            for (int i = 0; i <= P; ++i)
                #pragma unroll
                for (int j = 0; j <= P; ++j) S[i][j] = 0.0;
            int idx = 0;
            #pragma unroll
            for (int p = 0; p <= P; ++p)
                #pragma unroll
                for (int i = 0; i <= p; ++i)
                    #pragma unroll
                    for (int j = 0; j <= p - i; ++j, ++idx)
                        if (idx < NC) S[i][j] = fma(__ldg(coeffs + idx), M[2][p - i - j][k3], S[i][j]);
            #pragma unroll 1
            for (int k2 = 0; k2 <= P; ++k2)
            {
                double R[N];                                // R[a] = sum_b S[a][b] My[b][k2]
                #pragma unroll
                for (int i = 0; i <= P; ++i)
                {
                    double r = 0.0;
                    #pragma unroll
                    for (int j = 0; j <= P - i; ++j) r = fma(S[i][j], M[1][j][k2], r);
                    R[i] = r;
                }
                #pragma unroll 1
                for (int k1 = 0; k1 <= P; ++k1)
                {
                    double b = 0.0;
                    #pragma unroll
                    for (int i = 0; i <= P; ++i) b = fma(R[i], M[0][i][k1], b);
                    mn = fmin(mn, b); mx = fmax(mx, b);
                }
            }
        }
        const double allow = __dmul_ru(ldexp(1.0, kBoundsKappaLog2[P] - 53), sAbs);
        return make_double2(__dsub_rd(mn, allow), __dadd_ru(mx, allow));
    }

    __device__ double2 leafHullAny(const double* __restrict__ coeffs, int degree, int depth, const double (&ua)[3], const double (&ub)[3])
    {
        switch (degree)
        {
            case 0:  return leafHull<0>(coeffs, depth, ua, ub);
            case 1:  return leafHull<1>(coeffs, depth, ua, ub);
            case 2:  return leafHull<2>(coeffs, depth, ua, ub);
            case 3:  return leafHull<3>(coeffs, depth, ua, ub);
            case 4:  return leafHull<4>(coeffs, depth, ua, ub);
            case 5:  return leafHull<5>(coeffs, depth, ua, ub);
            case 6:  return leafHull<6>(coeffs, depth, ua, ub);
            case 7:  return leafHull<7>(coeffs, depth, ua, ub);
            case 8:  return leafHull<8>(coeffs, depth, ua, ub);
            case 9:  return leafHull<9>(coeffs, depth, ua, ub);
            case 10: return leafHull<10>(coeffs, depth, ua, ub);
            case 11: return leafHull<11>(coeffs, depth, ua, ub);
            default: return leafHull<12>(coeffs, depth, ua, ub);
        }
    }

    // Interval of a leaf over [lo, hi] (unit-cube coordinates, inside E(leaf)) at integer cell coordinates (x | y << 10 | z << 20).
    __device__ __forceinline__ double2 leafHullBox(const DeviceTreeView& view, uint4 raw, uint32_t cell, const double (&lo)[3],
                                                   const double (&hi)[3])
    {
        const int d = (int)raw.w;
        const double scale = (double)(2u << d);
        double ua[3], ub[3];
        for (int a = 0; a < 3; ++a)
        {
            double elo, ehi, c;
            boundsCell(d, (cell >> (10 * a)) & 1023u, elo, ehi, c);
            ua[a] = (lo[a] - c) * scale; ub[a] = (hi[a] - c) * scale;
        }
        return leafHullAny(view.coeffs + raw.y, (int)raw.z, d, ua, ub);
    }

    // Table pass over the nodes of depth d: a leaf's entry is its interval over E(leaf); an internal node hands its children
    // their cell coordinates.
    __global__ void __launch_bounds__(128) boundsLeafTableKernel(const DeviceTreeView view, int d, uint32_t* __restrict__ cells,
                                                                 double2* __restrict__ table)
    {
        const uint32_t node = blockIdx.x * blockDim.x + threadIdx.x;
        if (node >= view.nNodes) return;
        const uint4 raw = __ldg(reinterpret_cast<const uint4*>(view.nodes) + node);
        if ((int)raw.w != d) return;
        const uint32_t cell = cells[node];
        if (raw.z == kInternalTag)
        {
            for (uint32_t k = 0; k < 8; ++k)
            {
                uint32_t c = 0;
                for (int a = 0; a < 3; ++a) c |= ((((cell >> (10 * a)) & 1023u) << 1 | ((k >> a) & 1u)) << (10 * a));
                cells[raw.x + k] = c;
            }
            return;
        }
        double lo[3], hi[3];
        for (int a = 0; a < 3; ++a)
        {
            double c;
            boundsCell(d, (cell >> (10 * a)) & 1023u, lo[a], hi[a], c);
        }
        table[node] = leafHullBox(view, raw, cell, lo, hi);
    }

    // Table pass over the internal nodes of depth d (their children's entries are final): min and max of the 8 children.
    __global__ void __launch_bounds__(128) boundsInternalTableKernel(const DeviceTreeView view, int d, double2* __restrict__ table)
    {
        const uint32_t node = blockIdx.x * blockDim.x + threadIdx.x;
        if (node >= view.nNodes) return;
        const uint4 raw = __ldg(reinterpret_cast<const uint4*>(view.nodes) + node);
        if ((int)raw.w != d || raw.z != kInternalTag) return;
        double2 e = table[raw.x];
        for (uint32_t k = 1; k < 8; ++k)
        {
            const double2 c = table[raw.x + k];
            e.x = fmin(e.x, c.x); e.y = fmax(e.y, c.y);
        }
        table[node] = e;
    }

    __device__ __forceinline__ double warpMin(double v)
    {
        #pragma unroll
        for (int o = 16; o; o >>= 1) v = fmin(v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
        return v;
    }
    __device__ __forceinline__ double warpMax(double v)
    {
        #pragma unroll
        for (int o = 16; o; o >>= 1) v = fmax(v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
        return v;
    }

    // One box per warp, persistent grid; the warp's stack holds (node, cell coordinates) in shared memory.
    __global__ void __launch_bounds__(kBoundsThreads)
    boundsKernel(const DeviceTreeView view, const double2* __restrict__ table, const double* __restrict__ boxLo,
                 const double* __restrict__ boxHi, size_t n, double* __restrict__ fLo, double* __restrict__ fHi)
    {
        __shared__ uint2 sStack[kBoundsThreads / 32][kBoundsStack];
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        uint2* stack = sStack[warp];
        const size_t warpsTotal = (size_t)gridDim.x * (kBoundsThreads / 32);
        const double inf = __longlong_as_double(0x7FF0000000000000ll);
        for (size_t box = (size_t)blockIdx.x * (kBoundsThreads / 32) + warp; box < n; box += warpsTotal)
        {
            double plo[3], phi[3];
            bool bad = false, outside = false, partial = false;
            for (int a = 0; a < 3; ++a)
            {
                const double l = boxLo[3 * box + a], h = boxHi[3 * box + a];
                bad = bad || !(l <= h);                                          // NaN or inverted
                plo[a] = (l - view.map.centre[a]) * view.map.invSizes[a];       // Query's map (findLeaf)
                phi[a] = (h - view.map.centre[a]) * view.map.invSizes[a];
                outside = outside || phi[a] < -kBoundsL || plo[a] > kBoundsL;
                partial = partial || plo[a] < -kBoundsL || phi[a] > kBoundsL;
            }
            if (bad || outside)
            {
                if (lane == 0)
                {
                    const double v = bad ? __longlong_as_double(0x7FF8000000000000ll) : DBL_MAX;
                    fLo[box] = v; fHi[box] = v;
                }
                continue;
            }
            double runLo = inf, runHi = partial ? DBL_MAX : -inf;
            if (lane == 0) stack[0] = make_uint2(0u, 0u);
            int top = 1;
            __syncwarp();
            while (top > 0)
            {
                const int take = min(top, 32);
                top -= take;
                const bool have = lane < take;
                const uint2 e = have ? stack[top + lane] : make_uint2(0u, 0u);
                __syncwarp();
                double cLo = inf, cHi = -inf;
                bool push = false;
                uint4 raw = make_uint4(0u, 0u, 0u, 0u);
                if (have)
                {
                    raw = __ldg(reinterpret_cast<const uint4*>(view.nodes) + e.x);
                    const int d = (int)raw.w;
                    double lo[3], hi[3];
                    bool miss = false, covered = true;
                    for (int a = 0; a < 3; ++a)
                    {
                        double elo, ehi, c;
                        boundsCell(d, (e.y >> (10 * a)) & 1023u, elo, ehi, c);
                        miss = miss || phi[a] < elo || plo[a] > ehi;            // touching counts
                        covered = covered && plo[a] <= elo && phi[a] >= ehi;
                        lo[a] = fmax(plo[a], elo); hi[a] = fmin(phi[a], ehi);
                    }
                    if (!miss)
                    {
                        const double2 t = table[e.x];
                        if (t.x >= runLo && t.y <= runHi) {}                   // cannot change the result
                        else if (covered) { cLo = t.x; cHi = t.y; }
                        else if (raw.z == kInternalTag) push = true;
                        else
                        {
                            const double2 h = leafHullBox(view, raw, e.y, lo, hi);
                            cLo = fmax(h.x, t.x); cHi = fmin(h.y, t.y);
                        }
                    }
                }
                const unsigned pm = __ballot_sync(0xFFFFFFFFu, push);
                if (push)
                {
                    const int off = top + 8 * __popc(pm & ((1u << lane) - 1u));
                    for (uint32_t k = 0; k < 8; ++k)
                    {
                        uint32_t c = 0;
                        for (int a = 0; a < 3; ++a) c |= ((((e.y >> (10 * a)) & 1023u) << 1 | ((k >> a) & 1u)) << (10 * a));
                        stack[off + k] = make_uint2(raw.x + k, c);
                    }
                }
                top += 8 * __popc(pm);
                __syncwarp();
                runLo = fmin(runLo, warpMin(cLo));
                runHi = fmax(runHi, warpMax(cHi));
            }
            if (lane == 0) { fLo[box] = runLo; fHi[box] = runHi; }
        }
    }
}
