// raycast_kernels.cuh — hpsdf_raycast: the first crossing of F = iso along rays, found exactly per leaf (DESIGN §12).
//
// A ray x(t) = o + t d is mapped with Query's root map (p0 = (o - centre) invSizes, dp = d invSizes) and clipped to the unit
// cube: [ta, tb]. The walk locates leaves by integer cell coordinates at the finest level (1024 per axis): the top table takes
// the top four bits of each coordinate, then the QNode descent one bit per level. A leaf's box is exact in f64; the leaf's
// sub-interval ends at the smallest slab exit of the box (clamped to tb). The next point sets the crossed coordinate to the
// leaf's face exactly and clamps the other two into the box and against moving backwards, so every integer coordinate is
// monotone along the walk and a ray visits at most 3 * 1024 leaves, through edges, corners and face planes too.
//
// On a sub-interval the field is the leaf polynomial restricted to a segment: a univariate polynomial of degree <= m, with
// m the warp's largest leaf degree (warp-uniform control as in evalWarp). Its values g_j = P(u(tau_j)) - iso at the m+1
// Chebyshev-Lobatto nodes tau_j of [0, 1] (endpoints included) times the inverse Bernstein collocation matrix of those nodes
// (c_rayBern, built on the host) give its Bernstein coefficients; rows 0 and m are exact unit rows, so B_0 = g(0) and
// B_m = g(1) bit for bit. B_0 <= 0 is a hit at the start of the sub-interval; all B_j > 0 is no crossing (convex hull);
// otherwise a depth-first, left-first bisection names intervals by (level, index), recomputes their coefficients from the
// [0, 1] ones by two de Casteljau steps (no stack) and reports the left end of the first level-44 interval whose hull
// reaches 0.
#pragma once
#include "query_kernels.cuh"

namespace hpsdf
{
    constexpr int kRayRootLevels = 44;                    // bisection depth: intervals of 2^-44 of the sub-interval
    constexpr int kRayMaxVisits = 64 * kRayRootLevels;    // bisection intervals tested per leaf at most (near-touches backtrack)
    constexpr int kRayMaxSteps = 3 * 1024 + 3;            // leaves per ray at most: three monotone 10-bit coordinates
    __host__ __device__ constexpr int rayNodeOffset(int m) { return m * (m + 1) / 2; }                 // 91 nodes in all
    __host__ __device__ constexpr int rayBernOffset(int m) { return m * (m + 1) * (2 * m + 1) / 6; }   // 819 entries in all
    __constant__ double c_rayNodes[rayNodeOffset(kMaxDegree + 1)];
    __constant__ double c_rayBern[rayBernOffset(kMaxDegree + 1)];

    // Chebyshev-Lobatto nodes tau_j = sin^2(pi j / 2m) of [0, 1] and the inverses of the Bernstein collocation matrices
    // C[j][i] = binom(m, i) tau_j^i (1 - tau_j)^(m - i), by Gauss-Jordan elimination with partial pivoting in long double.
    inline void rayBuildTables(double nodes[rayNodeOffset(kMaxDegree + 1)], double bern[rayBernOffset(kMaxDegree + 1)])
    {
        for (int m = 0; m <= kMaxDegree; ++m)
        {
            const int n = m + 1;
            long double tau[kMaxDegree + 1], a[kMaxDegree + 1][2 * (kMaxDegree + 1)];
            for (int j = 0; j < n; ++j)
            {
                const long double s = m ? sinl(3.141592653589793238462643383279502884L * j / (2.0L * m)) : 0.0L;
                tau[j] = j == 0 ? 0.0L : j == m ? 1.0L : s * s;
                nodes[rayNodeOffset(m) + j] = (double)tau[j];
                long double binom = 1.0L;
                for (int i = 0; i < n; ++i)
                {
                    a[j][i] = binom * powl(tau[j], (long double)i) * powl(1.0L - tau[j], (long double)(m - i));
                    a[j][n + i] = i == j ? 1.0L : 0.0L;
                    binom = binom * (m - i) / (i + 1);
                }
            }
            for (int c = 0; c < n; ++c)
            {
                int piv = c;
                for (int r = c + 1; r < n; ++r) if (fabsl(a[r][c]) > fabsl(a[piv][c])) piv = r;
                for (int k = 0; k < 2 * n; ++k) { const long double x = a[c][k]; a[c][k] = a[piv][k]; a[piv][k] = x; }
                const long double d = a[c][c];
                for (int k = 0; k < 2 * n; ++k) a[c][k] /= d;
                for (int r = 0; r < n; ++r)
                    if (r != c)
                    {
                        const long double f = a[r][c];
                        for (int k = 0; k < 2 * n; ++k) a[r][k] -= f * a[c][k];
                    }
            }
            for (int i = 0; i < n; ++i)
                for (int j = 0; j < n; ++j)
                {
                    double v = (double)a[i][n + j];
                    if (i == 0 || i == m) v = (i == 0 ? j == 0 : j == m) ? 1.0 : 0.0;   // tau_0 = 0, tau_m = 1: exact unit rows
                    bern[rayBernOffset(m) + i * n + j] = v;
                }
        }
    }

    // Finest-level cell of a unit-cube coordinate, exactly: a coordinate on a cell face belongs to the upper cell (Query's
    // p >= c) unless the ray moves down that axis.
    __device__ __forceinline__ int rayCell(double p, double dp)
    {
        int i = (int)floor((p + 0.5) * 1024.0);
        i = min(max(i, 0), 1023);
        if (p < i * (1.0 / 1024.0) - 0.5) --i;
        else if (i < 1023 && p >= (i + 1) * (1.0 / 1024.0) - 0.5) ++i;
        if (dp < 0.0 && i > 0 && p == i * (1.0 / 1024.0) - 0.5) --i;
        return i;
    }

    // Bernstein coefficients of the restriction of c (on [0, 1]) to [i 2^-L, (i+1) 2^-L]: de Casteljau at the right end,
    // keep the left part, then at the left end of that part, keep the right part.
    template <int M>
    __device__ __forceinline__ void rayRestrict(const double (&c)[M + 1], uint64_t i, int L, double (&r)[M + 1])
    {
        #pragma unroll
        for (int j = 0; j <= M; ++j) r[j] = c[j];
        const double a = ldexp((double)i, -L), b = ldexp((double)(i + 1), -L);
        if (b < 1.0)
        {
            #pragma unroll
            for (int s = 1; s <= M; ++s)
                #pragma unroll
                for (int j = M; j >= s; --j) r[j] = fma(b, r[j], (1.0 - b) * r[j - 1]);
        }
        if (i)
        {
            const double s = a / b;
            #pragma unroll
            for (int k = 1; k <= M; ++k)
                #pragma unroll
                for (int j = 0; j <= M - k; ++j) r[j] = fma(s, r[j + 1], (1.0 - s) * r[j]);
        }
    }

    template <int M>
    __device__ __forceinline__ bool rayHullPositive(const double (&c)[M + 1])
    {
        bool pos = true;
        #pragma unroll
        for (int j = 0; j <= M; ++j) pos = pos && c[j] > 0.0;
        return pos;
    }

    // First root in [0, 1] of the polynomial with Bernstein coefficients B (B_0 > 0, some B_j <= 0): -1 when there is none.
    template <int M>
    __device__ double rayFirstRoot(const double (&B)[M + 1])
    {
        uint64_t i = 0;
        int L = 0;
        for (int visits = 0; visits < kRayMaxVisits; )
        {
            if (L == kRayRootLevels) break;                   // (L, i) reaches 0 within its hull: report its left end
            ++L; i <<= 1;
            for (;;)
            {
                double r[M + 1];
                rayRestrict<M>(B, i, L, r);
                ++visits;
                if (r[0] <= 0.0) return ldexp((double)i, -L);
                if (!rayHullPositive<M>(r) || visits == kRayMaxVisits) break;
                while (i & 1) { i >>= 1; --L; }               // excluded: the next interval in depth-first order
                if (L == 0) return -1.0;
                ++i;
            }
        }
        return ldexp((double)i, -L);
    }

    // One leaf sub-interval for the whole warp (all lanes call it; m = M is warp-uniform). Returns tau of the first point with
    // P <= iso on the lane's segment u_a -> u_b, or -1. Lanes without a leaf pass degree -1.
    template <int M>
    __device__ __forceinline__ double rayLeafFirstCrossing(const double* __restrict__ coeffs, int degree, int depth, const double (&ua)[3],
                                           const double (&ub)[3], double iso, bool pointOnly, const uint32_t* __restrict__ bidx)
    {
        double g[M + 1];
        #pragma unroll 1
        for (int j = 0; j <= M; ++j)
        {
            const double tau = c_rayNodes[rayNodeOffset(M) + j];
            double u[3];
            #pragma unroll
            for (int a = 0; a < 3; ++a) u[a] = j == 0 ? ua[a] : j == M ? ub[a] : fma(tau, ub[a] - ua[a], ua[a]);
            double v;
            if constexpr (M <= 6) v = evalLeafMasked<M>(coeffs, degree, u[0], u[1], u[2], depth);
            else v = degree < 0 ? 0.0 : evalLeafGeneric(coeffs, degree, u[0], u[1], u[2], depth, bidx);
            #pragma unroll
            for (int k = 0; k <= M; ++k) if (k == j) g[k] = v - iso;            // g stays in registers
        }
        if (degree < 0) return -1.0;
        if (g[0] <= 0.0) return 0.0;
        if constexpr (M == 0) return -1.0;
        else
        {
            if (pointOnly) return -1.0;
            double B[M + 1];
            B[0] = g[0]; B[M] = g[M];
            #pragma unroll
            for (int r = 1; r < M; ++r)
            {
                double s = 0.0;
                #pragma unroll
                for (int j = 0; j <= M; ++j) s = fma(c_rayBern[rayBernOffset(M) + r * (M + 1) + j], g[j], s);
                B[r] = s;
            }
            if (rayHullPositive<M>(B)) return -1.0;
            return rayFirstRoot<M>(B);
        }
    }

    // Degrees above 6 are rare: out of line, so that their 13-wide arrays do not set the register budget of the common path.
    template <int M>
    __device__ __noinline__ double rayLeafFirstCrossingHigh(const double* __restrict__ coeffs, int degree, int depth, const double (&ua)[3],
                                                            const double (&ub)[3], double iso, bool pointOnly, const uint32_t* __restrict__ bidx)
    {
        return rayLeafFirstCrossing<M>(coeffs, degree, depth, ua, ub, iso, pointOnly, bidx);
    }

    // Unit gradient of the leaf polynomial at local u, in user space (du/dx = 2^(depth+1) invSizes per axis), from the
    // derivative of the Legendre recurrence; (0, 0, 0) when it vanishes.
    __device__ __noinline__ void rayNormal(const double* __restrict__ coeffs, int degree, int depth, const double (&u)[3],
                                           const RootMap& map, const uint32_t* __restrict__ bidx, double (&nrm)[3])
    {
        LeafDerivs d;
        leafDerivsGeneric<1>(coeffs, degree, depth, u, bidx, d);
        double (&g)[3] = d.g;
        const double scale = (double)(2u << depth);
        for (int a = 0; a < 3; ++a) g[a] *= scale * map.invSizes[a];
        const double n = sqrt(g[0] * g[0] + (g[1] * g[1] + g[2] * g[2]));
        for (int a = 0; a < 3; ++a) nrm[a] = n > 0.0 && n <= DBL_MAX ? g[a] / n : 0.0;
    }

    struct RayArgs { double tMin, tMax, iso; };

    // One ray per lane, a warp per 32 consecutive rays, persistent grid. The top table is staged as in queryKernel.
    __global__ void __launch_bounds__(kQueryThreads, 2)
    raycastKernel(const DeviceTreeView view, const double* __restrict__ origins, const double* __restrict__ dirs, size_t n,
                  const RayArgs args, double* __restrict__ tHit, double* __restrict__ normals)
    {
        __shared__ uint32_t sTop[4096];
        const bool useTop = stageTop(sTop, view.top);
        const RootMap& map = view.map;
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const size_t nGroups = (n + 31) / 32, warpsTotal = (size_t)gridDim.x * (kQueryThreads / 32);
        for (size_t grp = (size_t)blockIdx.x * (kQueryThreads / 32) + warp; grp < nGroups; grp += warpsTotal)
        {
            const size_t ray = grp * 32 + lane;
            bool active = ray < n;
            double p0[3], dp[3], p[3], t = 0.0, tb = 0.0;
            int ix[3];
            if (active)
            {
                double ta = args.tMin;
                tb = args.tMax;
                bool dirOk = false;
                for (int a = 0; a < 3; ++a)
                {
                    const double o = origins[3 * ray + a], d = dirs[3 * ray + a];
                    p0[a] = (o - map.centre[a]) * map.invSizes[a];
                    dp[a] = d * map.invSizes[a];
                    active = active && isfinite(p0[a]) && isfinite(dp[a]);
                    dirOk = dirOk || dp[a] != 0.0;
                    if (dp[a] != 0.0)
                    {
                        const double t1 = (-0.5 - p0[a]) / dp[a], t2 = (0.5 - p0[a]) / dp[a];
                        ta = fmax(ta, fmin(t1, t2)); tb = fmin(tb, fmax(t1, t2));
                    }
                    else if (!(p0[a] >= -0.5 && p0[a] <= 0.5)) active = false;
                }
                active = active && dirOk && ta <= tb;
                t = ta;
                for (int a = 0; a < 3; ++a)
                    if (active) { p[a] = fmin(fmax(fma(ta, dp[a], p0[a]), -0.5), 0.5); ix[a] = rayCell(p[a], dp[a]); }
            }
            double tOut = __longlong_as_double(0x7FF0000000000000ll);       // +INFINITY: a miss
            const double* hitCoeffs = nullptr;
            int hitDeg = 0, hitDepth = 0;
            double hitU[3] = { 0.0, 0.0, 0.0 };
            for (int step = 0; __any_sync(0xFFFFFFFFu, active); ++step)
            {
                if (step == kRayMaxSteps) active = false;
                const double* coeffs = view.coeffs;
                int degree = -1, depth = 0, k = 0;
                double lo[3], hi[3], q[3], ua[3], ub[3], tExit = t;
                bool last = true;
                if (active)
                {
                    uint32_t cur = useTop ? sTop[(ix[0] >> 6) | ((ix[1] >> 6) << 4) | ((ix[2] >> 6) << 8)] : 0u;
                    uint4 raw = __ldg(reinterpret_cast<const uint4*>(view.nodes) + cur);
                    while (raw.z == kInternalTag)
                    {
                        const int s = 9 - (int)raw.w;
                        cur = raw.x + ((ix[0] >> s) & 1) + (((ix[1] >> s) & 1) << 1) + (((ix[2] >> s) & 1) << 2);
                        raw = __ldg(reinterpret_cast<const uint4*>(view.nodes) + cur);
                    }
                    degree = (int)raw.z; depth = (int)raw.w; coeffs = view.coeffs + raw.y;
                    const int sh = kMaxDepth - depth;
                    const double size = ldexp(1.0, -depth), scale = (double)(2u << depth);
                    tExit = tb;
                    k = -1;
                    for (int a = 0; a < 3; ++a)
                    {
                        lo[a] = ((ix[a] >> sh) << sh) * (1.0 / 1024.0) - 0.5;
                        hi[a] = lo[a] + size;
                        if (dp[a] != 0.0)
                        {
                            const double te = ((dp[a] > 0.0 ? hi[a] : lo[a]) - p0[a]) / dp[a];
                            if (te < tExit) { tExit = te; k = a; }
                        }
                    }
                    tExit = fmax(tExit, t);
                    last = k < 0;
                    for (int a = 0; a < 3; ++a)
                    {
                        double v = fmin(fmax(fma(tExit, dp[a], p0[a]), lo[a]), hi[a]);
                        v = dp[a] > 0.0 ? fmax(v, p[a]) : dp[a] < 0.0 ? fmin(v, p[a]) : p[a];
                        if (a == k) v = dp[a] > 0.0 ? hi[a] : lo[a];
                        q[a] = v;
                        const double c = lo[a] + 0.5 * size;
                        ua[a] = (p[a] - c) * scale; ub[a] = (q[a] - c) * scale;
                    }
                }
                const int m = (int)__reduce_max_sync(0xFFFFFFFFu, (unsigned)(degree < 0 ? 0 : degree));
                const bool pointOnly = tExit == t;
                double tau;
                switch (m)
                {
                    case 0:  tau = rayLeafFirstCrossing<0>(coeffs, degree, depth, ua, ub, args.iso, pointOnly, view.bidx); break;
                    case 1:  tau = rayLeafFirstCrossing<1>(coeffs, degree, depth, ua, ub, args.iso, pointOnly, view.bidx); break;
                    case 2:  tau = rayLeafFirstCrossing<2>(coeffs, degree, depth, ua, ub, args.iso, pointOnly, view.bidx); break;
                    case 3:  tau = rayLeafFirstCrossing<3>(coeffs, degree, depth, ua, ub, args.iso, pointOnly, view.bidx); break;
                    case 4:  tau = rayLeafFirstCrossing<4>(coeffs, degree, depth, ua, ub, args.iso, pointOnly, view.bidx); break;
                    case 5:  tau = rayLeafFirstCrossing<5>(coeffs, degree, depth, ua, ub, args.iso, pointOnly, view.bidx); break;
                    case 6:  tau = rayLeafFirstCrossing<6>(coeffs, degree, depth, ua, ub, args.iso, pointOnly, view.bidx); break;
                    case 7:  tau = rayLeafFirstCrossingHigh<7>(coeffs, degree, depth, ua, ub, args.iso, pointOnly, view.bidx); break;
                    case 8:  tau = rayLeafFirstCrossingHigh<8>(coeffs, degree, depth, ua, ub, args.iso, pointOnly, view.bidx); break;
                    case 9:  tau = rayLeafFirstCrossingHigh<9>(coeffs, degree, depth, ua, ub, args.iso, pointOnly, view.bidx); break;
                    case 10: tau = rayLeafFirstCrossingHigh<10>(coeffs, degree, depth, ua, ub, args.iso, pointOnly, view.bidx); break;
                    case 11: tau = rayLeafFirstCrossingHigh<11>(coeffs, degree, depth, ua, ub, args.iso, pointOnly, view.bidx); break;
                    default: tau = rayLeafFirstCrossingHigh<12>(coeffs, degree, depth, ua, ub, args.iso, pointOnly, view.bidx); break;
                }
                if (!active) continue;
                if (tau >= 0.0)
                {
                    tOut = tau == 0.0 ? t : fma(tau, tExit - t, t);
                    hitCoeffs = coeffs; hitDeg = degree; hitDepth = depth;
                    for (int a = 0; a < 3; ++a) hitU[a] = tau == 0.0 ? ua[a] : fma(tau, ub[a] - ua[a], ua[a]);
                    active = false;
                    continue;
                }
                if (last) { active = false; continue; }
                // step across face k into the next leaf
                const int sh = kMaxDepth - depth;
                const int nk = dp[k] > 0.0 ? ((ix[k] >> sh) + 1) << sh : ((ix[k] >> sh) << sh) - 1;
                if (nk < 0 || nk > 1023) { active = false; continue; }
                for (int a = 0; a < 3; ++a)
                {
                    p[a] = q[a];
                    ix[a] = a == k ? nk : rayCell(q[a], dp[a]);
                }
                t = tExit;
            }
            if (ray < n)
            {
                tHit[ray] = tOut;
                if (normals)
                {
                    double nv[3] = { 0.0, 0.0, 0.0 };
                    if (hitCoeffs) rayNormal(hitCoeffs, hitDeg, hitDepth, hitU, map, view.bidx, nv);
                    for (int a = 0; a < 3; ++a) normals[3 * ray + a] = nv[a];
                }
            }
        }
    }
}
