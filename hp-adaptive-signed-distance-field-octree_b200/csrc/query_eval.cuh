// query_eval.cuh — Octree::Query (Source/HP/Octree.cpp:662-702) and FApprox (:859-901) for one point, on the device.
//
// Reference: map the point into the unit cube with the f32-ROUNDED inverse root sizes (:323, :420, :665); reject it if
// its f32 cast is outside [-0.5, 0.5]^3 (:668-671, DBL_MAX); descend comparing the f64 coordinate with the f32 cell
// midpoint (:677-685); evaluate sum_i coeffs[i] * Lx[a_i] Ly[b_i] Lz[c_i] with Legendre recurrences scaled by
// NormalisedLengths[.][depth] in BasisIndexValues order.
//
// Here: cells are dyadic, so midpoints are tracked exactly in f64 instead of being loaded; the complete 16^3 grid of
// UniformlyRefine (:112-191) is entered through a 4096-entry table (shared-memory staged by the batch kernels) after four
// compare-only levels; nodes are 16-byte records (one LDG.128); coefficients sit in a padded store where every leaf is
// 16-byte aligned so they stream in as LDG.128 pairs; up to degree 6 the basis loop is unrolled with all Legendre values
// in registers, above it a loop over the basis table of the view. findLeaf is the one descent over QNodes (raycastKernel
// keeps its own integer-coordinate walk); evalWarp evaluates a warp's hits, treeQuery one thread's point with the same
// arithmetic.
#pragma once
#include <cfloat>
#include "hp_common.h"

namespace hpsdf
{
    // Derivatives of a leaf polynomial with respect to its local coordinate u: gradient, and Hessian in the order
    // xx, xy, xz, yy, yz, zz (filled for ORDER 2 only).
    struct LeafDerivs
    {
        double g[3] = { 0.0, 0.0, 0.0 };
        double h[6] = { 0.0, 0.0, 0.0, 0.0, 0.0, 0.0 };
    };

    // Warp-uniform evaluation: all lanes run the instantiation of the warp's LARGEST leaf degree and switch whole shells
    // off with a predicate (p <= myDeg), so lanes whose leaves have different degrees do not serialise (ncu showed 17 of
    // 32 lanes active per instruction when each lane branched to its own degree). Lanes without a leaf pass myDeg = -1.
    // ORDER 1 / 2 also accumulate the derivatives into *dv, from the derivatives of the Legendre recurrence
    // (P'_j = r0 (P_j-1 + u P'_j-1) - r1 P'_j-2, P''_j = r0 (2 P'_j-1 + u P''_j-1) - r1 P''_j-2). The value keeps ORDER 0's
    // products and order, and no product of it gets another use, so it is Query's to the bit.
    template <int DEG, int ORDER = 0>
    __device__ __forceinline__ double evalLeafMasked(const double* __restrict__ coeffs, int myDeg, double ux, double uy, double uz, int depth,
                                                     LeafDerivs* dv = nullptr)
    {
        constexpr int N1 = ORDER >= 1 ? DEG + 1 : 1, N2 = ORDER >= 2 ? DEG + 1 : 1;
        double lx[DEG + 1], ly[DEG + 1], lz[DEG + 1];
        double dlx[N1], dly[N1], dlz[N1], ddlx[N2], ddly[N2], ddlz[N2];
        {
            const double nl0 = c_nl[0][depth];
            lx[0] = nl0; ly[0] = nl0; lz[0] = nl0;
            if constexpr (ORDER >= 1) { dlx[0] = 0.0; dly[0] = 0.0; dlz[0] = 0.0; }
            if constexpr (ORDER >= 2) { ddlx[0] = 0.0; ddly[0] = 0.0; ddlz[0] = 0.0; }
            double ax2 = 0.0, ax1 = 1.0, ay2 = 0.0, ay1 = 1.0, az2 = 0.0, az1 = 1.0;
            double bx2 = 0.0, bx1 = 0.0, by2 = 0.0, by1 = 0.0, bz2 = 0.0, bz1 = 0.0;      // P'
            double cx2 = 0.0, cx1 = 0.0, cy2 = 0.0, cy1 = 0.0, cz2 = 0.0, cz1 = 0.0;      // P''
            #pragma unroll
            for (int j = 1; j <= DEG; ++j)
            {
                const double r0 = c_rec[j][0], r1 = c_rec[j][1], nl = c_nl[j][depth];
                if constexpr (ORDER >= 2)
                {
                    const double cx = r0 * (2.0 * bx1 + ux * cx1) - r1 * cx2; cx2 = cx1; cx1 = cx; ddlx[j] = cx * nl;
                    const double cy = r0 * (2.0 * by1 + uy * cy1) - r1 * cy2; cy2 = cy1; cy1 = cy; ddly[j] = cy * nl;
                    const double cz = r0 * (2.0 * bz1 + uz * cz1) - r1 * cz2; cz2 = cz1; cz1 = cz; ddlz[j] = cz * nl;
                }
                if constexpr (ORDER >= 1)
                {
                    const double bx = r0 * (ax1 + ux * bx1) - r1 * bx2; bx2 = bx1; bx1 = bx; dlx[j] = bx * nl;
                    const double by = r0 * (ay1 + uy * by1) - r1 * by2; by2 = by1; by1 = by; dly[j] = by * nl;
                    const double bz = r0 * (az1 + uz * bz1) - r1 * bz2; bz2 = bz1; bz1 = bz; dlz[j] = bz * nl;
                }
                const double ax = r0 * ux * ax1 - r1 * ax2; ax2 = ax1; ax1 = ax; lx[j] = ax * nl;      // Octree.cpp:879-883
                const double ay = r0 * uy * ay1 - r1 * ay2; ay2 = ay1; ay1 = ay; ly[j] = ay * nl;
                const double az = r0 * uz * az1 - r1 * az2; az2 = az1; az1 = az; lz[j] = az * nl;
            }
        }
        const double2* c2 = reinterpret_cast<const double2*>(coeffs);
        double f = 0.0;
        int idx = 0;
        double2 cur = make_double2(0.0, 0.0);
        #pragma unroll
        for (int p = 0; p <= DEG; ++p)
        {
            const bool on = p <= myDeg;
            #pragma unroll
            for (int i = 0; i <= p; ++i)
            {
                #pragma unroll
                for (int j = 0; j <= p - i; ++j)
                {
                    const int k = p - i - j;
                    // the reference stores 83 coefficients for a degree-6 leaf: (6,0,0) exists only from degree 7 on
                    const bool term = on && !(idx == 83 && myDeg == 6);
                    if ((idx & 1) == 0) { if (on) cur = __ldg(c2 + (idx >> 1)); }
                    const double cv = (idx & 1) ? cur.y : cur.x;
                    if (term) f = fma(cv, (lx[i] * ly[j]) * lz[k], f);                                  // Octree.cpp:891-897
                    if constexpr (ORDER >= 1)
                        if (term)
                        {
                            dv->g[0] = fma(cv, (dlx[i] * ly[j]) * lz[k], dv->g[0]);
                            dv->g[1] = fma(cv, (lx[i] * dly[j]) * lz[k], dv->g[1]);
                            dv->g[2] = fma(cv, (lx[i] * ly[j]) * dlz[k], dv->g[2]);
                        }
                    if constexpr (ORDER >= 2)
                        if (term)
                        {
                            dv->h[0] = fma(cv, (ddlx[i] * ly[j]) * lz[k], dv->h[0]);
                            dv->h[1] = fma(cv, (dlx[i] * dly[j]) * lz[k], dv->h[1]);
                            dv->h[2] = fma(cv, (dlx[i] * ly[j]) * dlz[k], dv->h[2]);
                            dv->h[3] = fma(cv, (lx[i] * ddly[j]) * lz[k], dv->h[3]);
                            dv->h[4] = fma(cv, (lx[i] * dly[j]) * dlz[k], dv->h[4]);
                            dv->h[5] = fma(cv, (lx[i] * ly[j]) * ddlz[k], dv->h[5]);
                        }
                    ++idx;
                }
            }
        }
        return f;
    }

    // Degrees above 6 are rare: a loop over the basis table with the Legendre values in local memory keeps the register
    // count of the kernel set by the common degrees.
    __device__ __noinline__ double evalLeafGeneric(const double* __restrict__ coeffs, int degree, double ux, double uy, double uz,
                                                   int depth, const uint32_t* __restrict__ bidx)
    {
        double l[3][kMaxDegree + 1];
        const double u[3] = { ux, uy, uz };
        for (int a = 0; a < 3; ++a)
        {
            l[a][0] = c_nl[0][depth];
            double m2 = 0.0, m1 = 1.0;
            for (int j = 1; j <= degree; ++j)
            {
                const double v = c_rec[j][0] * u[a] * m1 - c_rec[j][1] * m2; m2 = m1; m1 = v;
                l[a][j] = v * c_nl[j][depth];
            }
        }
        double f = 0.0;
        const int n = coeffCount(degree);
        for (int i = 0; i < n; ++i)
        {
            const uint32_t abc = __ldg(bidx + i);
            f = fma(coeffs[i], (l[0][abc & 0xFF] * l[1][(abc >> 8) & 0xFF]) * l[2][(abc >> 16) & 0xFF], f);
        }
        return f;
    }

    // Gradient and, for ORDER 2, Hessian of a leaf polynomial of any degree with respect to its local u: the basis-table loop
    // over Legendre values and their derivatives in local memory. rayNormal is this routine (ORDER 1) plus normalisation.
    template <int ORDER>
    __device__ __noinline__ void leafDerivsGeneric(const double* __restrict__ coeffs, int degree, int depth, const double (&u)[3],
                                                   const uint32_t* __restrict__ bidx, LeafDerivs& d)
    {
        constexpr int N2 = ORDER >= 2 ? kMaxDegree + 1 : 1;
        double l[3][kMaxDegree + 1], dl[3][kMaxDegree + 1], ddl[3][N2];
        for (int a = 0; a < 3; ++a)
        {
            l[a][0] = c_nl[0][depth]; dl[a][0] = 0.0;
            if constexpr (ORDER >= 2) ddl[a][0] = 0.0;
            double m2 = 0.0, m1 = 1.0, d2 = 0.0, d1 = 0.0, e2 = 0.0, e1 = 0.0;
            for (int j = 1; j <= degree; ++j)
            {
                const double r0 = c_rec[j][0], r1 = c_rec[j][1];
                if constexpr (ORDER >= 2)
                {
                    const double ev = r0 * (2.0 * d1 + u[a] * e1) - r1 * e2;
                    e2 = e1; e1 = ev;
                    ddl[a][j] = ev * c_nl[j][depth];
                }
                const double v = r0 * u[a] * m1 - r1 * m2, dv = r0 * (m1 + u[a] * d1) - r1 * d2;
                m2 = m1; m1 = v; d2 = d1; d1 = dv;
                l[a][j] = v * c_nl[j][depth]; dl[a][j] = dv * c_nl[j][depth];
            }
        }
        const int nc = coeffCount(degree);
        for (int i = 0; i < nc; ++i)
        {
            const uint32_t abc = __ldg(bidx + i);
            const int x = abc & 0xFF, y = (abc >> 8) & 0xFF, z = (abc >> 16) & 0xFF;
            const double c = __ldg(coeffs + i);
            d.g[0] = fma(c, (dl[0][x] * l[1][y]) * l[2][z], d.g[0]);
            d.g[1] = fma(c, (l[0][x] * dl[1][y]) * l[2][z], d.g[1]);
            d.g[2] = fma(c, (l[0][x] * l[1][y]) * dl[2][z], d.g[2]);
            if constexpr (ORDER >= 2)
            {
                d.h[0] = fma(c, (ddl[0][x] * l[1][y]) * l[2][z], d.h[0]);
                d.h[1] = fma(c, (dl[0][x] * dl[1][y]) * l[2][z], d.h[1]);
                d.h[2] = fma(c, (dl[0][x] * l[1][y]) * dl[2][z], d.h[2]);
                d.h[3] = fma(c, (l[0][x] * ddl[1][y]) * l[2][z], d.h[3]);
                d.h[4] = fma(c, (l[0][x] * dl[1][y]) * dl[2][z], d.h[4]);
                d.h[5] = fma(c, (l[0][x] * l[1][y]) * ddl[2][z], d.h[5]);
            }
        }
    }

    struct LeafHit
    {
        const double* coeffs = nullptr;
        double ux = 0.0, uy = 0.0, uz = 0.0;
        int    degree = -1;   // -1: no point, or the point is outside the root
        int    depth = 0;
    };

    // Octree::Query up to the leaf: root map, f32 containment test, descent (Octree.cpp:662-702). `top` is the view's
    // depth-4 table or a shared-memory copy of it, or nullptr to start at the root.
    __device__ __forceinline__ LeafHit findLeaf(const DeviceTreeView& view, const uint32_t* top, double x, double y, double z)
    {
        LeafHit h;
        const double px = (x - view.map.centre[0]) * view.map.invSizes[0];          // Octree.cpp:665
        const double py = (y - view.map.centre[1]) * view.map.invSizes[1];
        const double pz = (z - view.map.centre[2]) * view.map.invSizes[2];
        const float fx = (float)px, fy = (float)py, fz = (float)pz;       // Octree.cpp:668: contains() on the f32 cast, inclusive
        if (!(fx >= -0.5f && fx <= 0.5f && fy >= -0.5f && fy <= 0.5f && fz >= -0.5f && fz <= 0.5f)) return h;
        double cx = 0.0, cy = 0.0, cz = 0.0, q = 0.25;                    // centre of the current node, quarter of its size
        uint32_t cur = 0;
        if (top)
        {
            uint32_t code = 0;
            #pragma unroll
            for (int l = 0; l < kCoarseDepth; ++l)
            {
                const uint32_t bx = px >= cx, by = py >= cy, bz = pz >= cz;         // Octree.cpp:681-683
                cx += bx ? q : -q; cy += by ? q : -q; cz += bz ? q : -q; q *= 0.5;
                code = (code << 1) | bx | (by << 4) | (bz << 8);                    // x bits in [0,4), y in [4,8), z in [8,12)
            }
            cur = top[code & 0xFFF];
        }
        uint4 raw = __ldg(reinterpret_cast<const uint4*>(view.nodes) + cur);
        while (raw.z == kInternalTag)                                               // Octree.cpp:687
        {
            const uint32_t bx = px >= cx, by = py >= cy, bz = pz >= cz;
            cx += bx ? q : -q; cy += by ? q : -q; cz += bz ? q : -q; q *= 0.5;
            cur = raw.x + bx + (by << 1) + (bz << 2);                               // Octree.cpp:685
            raw = __ldg(reinterpret_cast<const uint4*>(view.nodes) + cur);
        }
        const double scale = (double)(2u << raw.w);                                 // Octree.cpp:862
        h.coeffs = view.coeffs + raw.y; h.degree = (int)raw.z; h.depth = (int)raw.w;
        h.ux = (px - cx) * scale; h.uy = (py - cy) * scale; h.uz = (pz - cz) * scale;
        return h;
    }

    // FApprox of a hit with the instantiation for degree m >= h.degree: the unrolled form up to 6, the basis-table loop above.
    // Both form the same products in the same order, so a lane's value does not depend on the degrees of the rest of its warp.
    __device__ __forceinline__ double evalHit(const LeafHit& h, int m, const uint32_t* __restrict__ bidx)
    {
        double v;
        switch (m)
        {
            case 0:  v = evalLeafMasked<0>(h.coeffs, h.degree, h.ux, h.uy, h.uz, h.depth); break;
            case 1:  v = evalLeafMasked<1>(h.coeffs, h.degree, h.ux, h.uy, h.uz, h.depth); break;
            case 2:  v = evalLeafMasked<2>(h.coeffs, h.degree, h.ux, h.uy, h.uz, h.depth); break;
            case 3:  v = evalLeafMasked<3>(h.coeffs, h.degree, h.ux, h.uy, h.uz, h.depth); break;
            case 4:  v = evalLeafMasked<4>(h.coeffs, h.degree, h.ux, h.uy, h.uz, h.depth); break;
            case 5:  v = evalLeafMasked<5>(h.coeffs, h.degree, h.ux, h.uy, h.uz, h.depth); break;
            case 6:  v = evalLeafMasked<6>(h.coeffs, h.degree, h.ux, h.uy, h.uz, h.depth); break;
            default: v = h.degree < 0 ? 0.0 : evalLeafGeneric(h.coeffs, h.degree, h.ux, h.uy, h.uz, h.depth, bidx); break;
        }
        return h.degree < 0 ? DBL_MAX : v;                                          // Octree.cpp:668-671
    }

    // Evaluate the hits of a whole warp (all 32 lanes must call this).
    __device__ __forceinline__ double evalWarp(const LeafHit& h, const uint32_t* __restrict__ bidx)
    {
        return evalHit(h, (int)__reduce_max_sync(0xFFFFFFFFu, (unsigned)(h.degree < 0 ? 0 : h.degree)), bidx);
    }

    // hpsdf_query for one point of one thread, with the arithmetic evalWarp gives its lane.
    __device__ __forceinline__ double treeQuery(const DeviceTreeView& tree, double x, double y, double z)
    {
        const LeafHit h = findLeaf(tree, tree.top, x, y, z);
        return evalHit(h, h.degree, tree.bidx);
    }
}
