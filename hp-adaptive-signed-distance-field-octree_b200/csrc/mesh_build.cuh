// mesh_build.cuh — hpsdf_mesh_create on the device: everything Meshing::Mesh + Meshing::BVH set up on the host in the
// reference (and in round 1 of this library), as kernels over the uploaded vertex / index arrays.
//
//   half-edge twins   Mesh::CreateHalfEdges (Source/Meshing/Mesh.cpp:87-131) looks every directed edge up in a std::map.
//                     Here: one radix sort of the 3n half-edges by their UNDIRECTED edge (stable, so each run is in half-edge
//                     order), then one thread per run replays the map's find / insert sequence restricted to that edge — the
//                     same twins, including the reference's first-occurrence rule on non-manifold input; an unpaired edge
//                     fails the mesh (:121-128).
//   pseudonormals     PseudoNormalFace / Edge / Vertex (Mesh.cpp:185-242), one thread per triangle, float32 with the reference's
//                     operation order and no FMA contraction; the angle weights use acosfExact, the fdlibm float algorithm,
//                     which returns the bits of the host libm's acosf for every float in [-1, 1] (tools/verify_acosf.c) — they
//                     decide signs, so the mesh distances stay bit-identical to the reference.
//   BVH               median split on the longest axis of the centroid bounds, <= 4 triangles per leaf, as a level-synchronous
//                     build: per level one stable radix sort of (segment, centroid coordinate on the segment's axis) keeps every
//                     segment in place and orders it, then segments split at their middle. The node numbering is the pre-order
//                     one (node, left subtree, right subtree); it depends on the triangle count alone. Bounds by a bottom-up
//                     refit; oriented boxes (frame of the mean normal) one warp per node; 4-wide collapse for meshSampleKernel.
//                     The reference's bottom-up pairing through an NNOctree (BVH.cpp:26-260) is not reproduced: any BVH gives
//                     the same closest triangle.
#pragma once
#include <cub/cub.cuh>
#include "hp_common.h"
#include "mesh_eval.cuh"

namespace hpsdf
{
    // ---- exact float arc cosine ------------------------------------------------------------------------------------------------
    __device__ __forceinline__ float acosfExact(float x)
    {
        const float one = 1.0f, pi = 3.1415925026e+00f, pio2_hi = 1.5707962513e+00f, pio2_lo = 7.5497894159e-08f,
                    pS0 = 1.6666667163e-01f, pS1 = -3.2556581497e-01f, pS2 = 2.0121252537e-01f, pS3 = -4.0055535734e-02f,
                    pS4 = 7.9153501429e-04f, pS5 = 3.4793309169e-05f,
                    qS1 = -2.4033949375e+00f, qS2 = 2.0209457874e+00f, qS3 = -6.8828397989e-01f, qS4 = 7.7038154006e-02f;
        const int hx = __float_as_int(x), ix = hx & 0x7fffffff;
        #define HP_M(a, b) __fmul_rn((a), (b))
        #define HP_A(a, b) __fadd_rn((a), (b))
        #define HP_S(a, b) __fsub_rn((a), (b))
        if (ix == 0x3f800000) return hx > 0 ? 0.0f : HP_A(pi, HP_M(2.0f, pio2_lo));
        if (ix > 0x3f800000) return __fdiv_rn(HP_S(x, x), HP_S(x, x));
        if (ix < 0x3f000000)
        {
            if (ix <= 0x23000000) return HP_A(pio2_hi, pio2_lo);
            const float z = HP_M(x, x);
            const float p = HP_M(z, HP_A(pS0, HP_M(z, HP_A(pS1, HP_M(z, HP_A(pS2, HP_M(z, HP_A(pS3, HP_M(z, HP_A(pS4, HP_M(z, pS5)))))))))));
            const float q = HP_A(one, HP_M(z, HP_A(qS1, HP_M(z, HP_A(qS2, HP_M(z, HP_A(qS3, HP_M(z, qS4))))))));
            const float r = __fdiv_rn(p, q);
            return HP_S(pio2_hi, HP_S(x, HP_S(pio2_lo, HP_M(x, r))));
        }
        if (hx < 0)
        {
            const float z = HP_M(HP_A(one, x), 0.5f);
            const float p = HP_M(z, HP_A(pS0, HP_M(z, HP_A(pS1, HP_M(z, HP_A(pS2, HP_M(z, HP_A(pS3, HP_M(z, HP_A(pS4, HP_M(z, pS5)))))))))));
            const float q = HP_A(one, HP_M(z, HP_A(qS1, HP_M(z, HP_A(qS2, HP_M(z, HP_A(qS3, HP_M(z, qS4))))))));
            const float s = __fsqrt_rn(z);
            const float r = __fdiv_rn(p, q);
            const float w = HP_S(HP_M(r, s), pio2_lo);
            return HP_S(pi, HP_M(2.0f, HP_A(s, w)));
        }
        const float z = HP_M(HP_S(one, x), 0.5f);
        const float s = __fsqrt_rn(z);
        const float df = __int_as_float(__float_as_int(s) & 0xfffff000);
        const float c = __fdiv_rn(HP_S(z, HP_M(df, df)), HP_A(s, df));
        const float p = HP_M(z, HP_A(pS0, HP_M(z, HP_A(pS1, HP_M(z, HP_A(pS2, HP_M(z, HP_A(pS3, HP_M(z, HP_A(pS4, HP_M(z, pS5)))))))))));
        const float q = HP_A(one, HP_M(z, HP_A(qS1, HP_M(z, HP_A(qS2, HP_M(z, HP_A(qS3, HP_M(z, qS4))))))));
        const float r = __fdiv_rn(p, q);
        const float w = HP_A(HP_M(r, s), c);
        return HP_M(2.0f, HP_A(df, w));
        #undef HP_M
        #undef HP_A
        #undef HP_S
    }

    __device__ __forceinline__ F3 normalized3(const F3& a)
    {
        const float z = dot3(a, a);
        if (z > 0.0f) { const float n = __fsqrt_rn(z); return f3(__fdiv_rn(a.x, n), __fdiv_rn(a.y, n), __fdiv_rn(a.z, n)); }
        return a;
    }

    struct MeshBuildIn
    {
        const float*    v;        // 3 floats per vertex
        const uint32_t* tri;      // 3 indices per triangle
        uint32_t        nVerts, nTris;
    };

    __device__ __forceinline__ F3 vertOf(const MeshBuildIn& M, uint32_t t, uint32_t k)
    {
        const uint32_t i = M.tri[3 * t + k];
        return f3(M.v[3 * (size_t)i], M.v[3 * (size_t)i + 1], M.v[3 * (size_t)i + 2]);
    }
    // PseudoNormalFace (Mesh.cpp:185-193)
    __device__ __forceinline__ F3 faceNormalOf(const MeshBuildIn& M, uint32_t t)
    {
        const F3 a = vertOf(M, t, 0);
        return normalized3(cross3(sub3(vertOf(M, t, 1), a), sub3(vertOf(M, t, 2), a)));
    }

    // ---- half-edges --------------------------------------------------------------------------------------------------------------
    __global__ void __launch_bounds__(256) meshEdgeKeysKernel(const MeshBuildIn M, const int vertexBits, unsigned long long* __restrict__ keys,
                                                              uint32_t* __restrict__ vals, uint32_t* __restrict__ he, uint32_t* __restrict__ flags)
    {
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= 3u * M.nTris) return;
        const uint32_t from = M.tri[i], to = (i % 3u == 2u) ? M.tri[i - 2] : M.tri[i + 1];
        if (from >= M.nVerts) atomicOr(flags, 1u);                                   // triangle index out of range
        const uint32_t lo = from < to ? from : to, hi = from < to ? to : from;
        keys[i] = ((unsigned long long)lo << vertexBits) | hi;                      // 2 * vertexBits significant bits: fewer radix passes
        vals[i] = i;
        he[i] = 0xFFFFFFFFu;
    }

    // One thread per run of equal undirected edges (sorted, half-edge order inside the run): the find / insert sequence of the
    // reference's std::map for the two directed keys of this edge (Mesh.cpp:96-118): "is the reverse edge known? pair with it :
    // remember this edge unless an equal one is already known".
    __global__ void __launch_bounds__(256) meshPairKernel(const MeshBuildIn M, const int vertexBits, const unsigned long long* __restrict__ keys,
                                                          const uint32_t* __restrict__ vals, uint32_t* __restrict__ he)
    {
        const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x, n = 3u * M.nTris;
        if (p >= n) return;
        const unsigned long long key = keys[p];
        if (p > 0 && keys[p - 1] == key) return;                                     // not the start of a run
        const uint32_t lo = (uint32_t)(key >> vertexBits);
        uint32_t stored[2] = { 0xFFFFFFFFu, 0xFFFFFFFFu };                           // first half-edge known per direction: [0] lo -> hi, [1] hi -> lo
        for (uint32_t q = p; q < n && keys[q] == key; ++q)
        {
            const uint32_t i = vals[q];
            const uint32_t dir = M.tri[i] == lo ? 0u : 1u;
            if (stored[dir ^ 1u] != 0xFFFFFFFFu) { he[stored[dir ^ 1u]] = i; he[i] = stored[dir ^ 1u]; }
            else if (stored[dir] == 0xFFFFFFFFu) stored[dir] = i;
        }
    }

    __global__ void __launch_bounds__(256) meshCheckPairedKernel(const uint32_t* __restrict__ he, uint32_t n, uint32_t* __restrict__ flags)
    {
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i < n && he[i] == 0xFFFFFFFFu) atomicOr(flags, 2u);                      // an edge without a twin: not a closed manifold
    }

    // ---- pseudonormals: 21 floats per triangle = face | edge AB, BC, CA | vertex A, B, C ----------------------------------------------
    __global__ void __launch_bounds__(128) meshPseudoKernel(const MeshBuildIn M, const uint32_t* __restrict__ he, float* __restrict__ pseudo)
    {
        const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
        if (t >= M.nTris) return;
        float* p = pseudo + 21 * (size_t)t;
        const F3 f = faceNormalOf(M, t);
        p[0] = f.x; p[1] = f.y; p[2] = f.z;
        const float PI = (float)3.14159265359;
        for (uint32_t s = 0; s < 3; ++s)
        {
            // PseudoNormalEdge (Mesh.cpp:196-213): nA * PI + nB * PI, normalised
            const uint32_t adjEdge = he[3 * t + s];
            const uint32_t adjTri = (adjEdge - (adjEdge % 3u)) / 3u;
            const F3 e = normalized3(add3(scale3(f, PI), scale3(faceNormalOf(M, adjTri), PI)));
            p[3 + 3 * s] = e.x; p[4 + 3 * s] = e.y; p[5 + 3 * s] = e.z;
            // PseudoNormalVertex (Mesh.cpp:216-242): walk the fan he -> next(twin(he)) until back at the start triangle
            F3 n = f3(0.0f, 0.0f, 0.0f);
            uint32_t curHE = 3 * t + s, curTri = t, guard = 0;
            do
            {
                const F3 c0 = vertOf(M, curTri, curHE % 3u), c1 = vertOf(M, curTri, (curHE + 1u) % 3u), c2 = vertOf(M, curTri, (curHE + 2u) % 3u);
                const float ang = acosfExact(dot3(normalized3(sub3(c1, c0)), normalized3(sub3(c2, c0))));
                n = add3(n, scale3(faceNormalOf(M, curTri), ang));
                curHE = he[curHE];
                curHE = ((curHE % 3u) == 2u) ? (curHE - 2u) : (curHE + 1u);
                curTri = (curHE - (curHE % 3u)) / 3u;
            } while (curTri != t && ++guard < 100000u);
            const F3 w = normalized3(n);
            p[12 + 3 * s] = w.x; p[13 + 3 * s] = w.y; p[14 + 3 * s] = w.z;
        }
    }

    // ---- BVH ---------------------------------------------------------------------------------------------------------------------
    __device__ __forceinline__ uint32_t orderedFloat(float x)
    {
        const uint32_t b = __float_as_uint(x + 0.0f);                 // -0 -> +0
        return b ^ ((b >> 31) ? 0xFFFFFFFFu : 0x80000000u);
    }
    __device__ __forceinline__ float unorderedFloat(uint32_t u)
    {
        return __uint_as_float(u ^ ((u >> 31) ? 0x80000000u : 0xFFFFFFFFu));
    }

    // per triangle: bounds and the centroid of the bounds (as the host builder of round 1: 0.5 * (min + max))
    __global__ void __launch_bounds__(256) meshTriBoundsKernel(const MeshBuildIn M, float* __restrict__ tmn, float* __restrict__ tmx, float* __restrict__ cen,
                                                               uint32_t* __restrict__ order, uint32_t* __restrict__ segBegin, uint32_t* __restrict__ segEnd,
                                                               uint32_t* __restrict__ segNode)
    {
        const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
        if (t >= M.nTris) return;
        const F3 a = vertOf(M, t, 0), b = vertOf(M, t, 1), c = vertOf(M, t, 2);
        const float mn[3] = { fminf(a.x, fminf(b.x, c.x)), fminf(a.y, fminf(b.y, c.y)), fminf(a.z, fminf(b.z, c.z)) };
        const float mx[3] = { fmaxf(a.x, fmaxf(b.x, c.x)), fmaxf(a.y, fmaxf(b.y, c.y)), fmaxf(a.z, fmaxf(b.z, c.z)) };
        for (int d = 0; d < 3; ++d) { tmn[3 * (size_t)t + d] = mn[d]; tmx[3 * (size_t)t + d] = mx[d]; cen[3 * (size_t)t + d] = 0.5f * (mn[d] + mx[d]); }
        order[t] = t; segBegin[t] = 0; segEnd[t] = M.nTris; segNode[t] = 0;
    }

    // number of nodes of the median-split tree over m triangles: from the table of the sizes that can occur (host, mesh.cpp)
    struct BvhCountTable { uint32_t n; uint32_t size[96]; uint32_t count[96]; };
    __device__ __forceinline__ uint32_t bvhNodeCountDev(const BvhCountTable& T, uint32_t m)
    {
        for (uint32_t i = 0; i < T.n; ++i) if (T.size[i] == m) return T.count[i];
        return 1u;
    }

    // centroid bounds of every active segment (segments longer than 4): block-aggregated when a block lies inside one segment
    __global__ void __launch_bounds__(256) meshSegBoundsKernel(const uint32_t* __restrict__ order, const uint32_t* __restrict__ segBegin,
                                                               const uint32_t* __restrict__ segEnd, const float* __restrict__ cen, uint32_t n,
                                                               uint32_t* __restrict__ cbounds /* 6 per position slot of the segment's begin */)
    {
        __shared__ uint32_t sLo[3], sHi[3];
        __shared__ int sUniform;
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        const bool valid = i < n;
        const uint32_t b = valid ? segBegin[i] : 0xFFFFFFFFu, e = valid ? segEnd[i] : 0u;
        const bool active = valid && e - b > 4u;
        uint32_t lo[3] = { 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu }, hi[3] = { 0u, 0u, 0u };
        if (active)
        {
            const uint32_t t = order[i];
            for (int d = 0; d < 3; ++d) lo[d] = hi[d] = orderedFloat(cen[3 * (size_t)t + d]);
        }
        if (threadIdx.x == 0) { sUniform = 1; for (int d = 0; d < 3; ++d) { sLo[d] = 0xFFFFFFFFu; sHi[d] = 0u; } }
        __syncthreads();
        const uint32_t first = segBegin[blockIdx.x * blockDim.x < n ? blockIdx.x * blockDim.x : n - 1];
        if (valid && b != first) sUniform = 0;
        __syncthreads();
        if (sUniform)
        {
            if (active) for (int d = 0; d < 3; ++d) { atomicMin(&sLo[d], lo[d]); atomicMax(&sHi[d], hi[d]); }
            __syncthreads();
            if (threadIdx.x < 3 && sHi[threadIdx.x] >= sLo[threadIdx.x])
            {
                atomicMin(cbounds + 6 * (size_t)first + threadIdx.x, sLo[threadIdx.x]);
                atomicMax(cbounds + 6 * (size_t)first + 3 + threadIdx.x, sHi[threadIdx.x]);
            }
        }
        else if (active)
            for (int d = 0; d < 3; ++d) { atomicMin(cbounds + 6 * (size_t)b + d, lo[d]); atomicMax(cbounds + 6 * (size_t)b + 3 + d, hi[d]); }
    }

    __global__ void __launch_bounds__(256) meshSegInitKernel(const uint32_t* __restrict__ segBegin, const uint32_t* __restrict__ segEnd, uint32_t n,
                                                             uint32_t* __restrict__ cbounds)
    {
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n || segBegin[i] != i || segEnd[i] - i <= 4u) return;
        for (int d = 0; d < 3; ++d) { cbounds[6 * (size_t)i + d] = 0xFFFFFFFFu; cbounds[6 * (size_t)i + 3 + d] = 0u; }
    }

    // sort key of every position: (segment begin, centroid coordinate on the segment's longest axis); finished segments keep
    // their order (begin = own position). The position that starts a segment also writes the segment's node.
    __global__ void __launch_bounds__(256) meshLevelKeysKernel(const uint32_t* __restrict__ order, const uint32_t* __restrict__ segBegin,
                                                               const uint32_t* __restrict__ segEnd, const uint32_t* __restrict__ segNode,
                                                               const float* __restrict__ cen, const uint32_t* __restrict__ cbounds, uint32_t n,
                                                               const BvhCountTable T, unsigned long long* __restrict__ keys, BvhNode* __restrict__ nodes,
                                                               uint32_t* __restrict__ parent, uint32_t* __restrict__ nodeDepth, uint32_t level)
    {
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n) return;
        const uint32_t b = segBegin[i], e = segEnd[i];
        if (e - b <= 4u)
        {
            keys[i] = ((unsigned long long)i << 32);
            if (i == b && e > b && segNode[i] != 0xFFFFFFFFu)
            {
                // a leaf that appears at this level (its node has not been written yet)
                BvhNode& nd = nodes[segNode[i]];
                if (nodeDepth[segNode[i]] == 0xFFFFFFFFu) { nd.a = b; nd.b = 0x80000000u | (e - b); nodeDepth[segNode[i]] = level; }
            }
            return;
        }
        const uint32_t* cb = cbounds + 6 * (size_t)b;
        const float ext[3] = { unorderedFloat(cb[3]) - unorderedFloat(cb[0]), unorderedFloat(cb[4]) - unorderedFloat(cb[1]), unorderedFloat(cb[5]) - unorderedFloat(cb[2]) };
        int axis = 0;
        if (ext[1] > ext[axis]) axis = 1;
        if (ext[2] > ext[axis]) axis = 2;
        keys[i] = ((unsigned long long)b << 32) | orderedFloat(cen[3 * (size_t)order[i] + axis]);
        if (i == b)
        {
            const uint32_t idx = segNode[i], mid = (b + e) / 2u;
            const uint32_t l = idx + 1u, r = idx + 1u + bvhNodeCountDev(T, mid - b);
            nodes[idx].a = l; nodes[idx].b = r;
            parent[l] = idx; parent[r] = idx;
            nodeDepth[idx] = level;
        }
    }

    // after the sort: every active segment splits at its middle
    __global__ void __launch_bounds__(256) meshLevelSplitKernel(uint32_t* __restrict__ segBegin, uint32_t* __restrict__ segEnd, uint32_t* __restrict__ segNode,
                                                                uint32_t n, const BvhCountTable T)
    {
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n) return;
        const uint32_t b = segBegin[i], e = segEnd[i];
        if (e - b <= 4u) return;
        const uint32_t idx = segNode[i], mid = (b + e) / 2u;
        if (i < mid) { segEnd[i] = mid; segNode[i] = idx + 1u; }
        else { segBegin[i] = mid; segNode[i] = idx + 1u + bvhNodeCountDev(T, mid - b); }
    }

    // leaves: bounds of their triangles; then every thread climbs: the second child to arrive at a node merges (bottom-up refit)
    __global__ void __launch_bounds__(256) meshRefitKernel(BvhNode* __restrict__ nodes, const uint32_t* __restrict__ parent, const uint32_t* __restrict__ order,
                                                           const float* __restrict__ tmn, const float* __restrict__ tmx, uint32_t nNodes,
                                                           uint32_t* __restrict__ arrived)
    {
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= nNodes) return;
        BvhNode nd = nodes[i];
        if (!(nd.b & 0x80000000u)) return;
        float mn[3] = { 3.4e38f, 3.4e38f, 3.4e38f }, mx[3] = { -3.4e38f, -3.4e38f, -3.4e38f };
        const uint32_t cnt = nd.b & 0x7FFFFFFFu;
        for (uint32_t k = 0; k < cnt; ++k)
        {
            const uint32_t t = order[nd.a + k];
            for (int d = 0; d < 3; ++d) { mn[d] = fminf(mn[d], tmn[3 * (size_t)t + d]); mx[d] = fmaxf(mx[d], tmx[3 * (size_t)t + d]); }
        }
        for (int d = 0; d < 3; ++d) { nodes[i].mn[d] = mn[d]; nodes[i].mx[d] = mx[d]; }
        uint32_t cur = i;
        while (cur != 0u)
        {
            const uint32_t par = parent[cur];
            __threadfence();
            if (atomicAdd(arrived + par, 1u) == 0u) return;              // the sibling subtree is not finished: its thread goes on
            const BvhNode p = nodes[par];
            const volatile BvhNode* L = nodes + p.a; const volatile BvhNode* R = nodes + p.b;
            for (int d = 0; d < 3; ++d)
            {
                nodes[par].mn[d] = fminf(L->mn[d], R->mn[d]);
                nodes[par].mx[d] = fmaxf(L->mx[d], R->mx[d]);
            }
            cur = par;
        }
    }

    // Oriented boxes (see mesh.cpp of round 1 for the rationale): one warp per node with at most 32 768 triangles. Frame =
    // area-weighted mean normal n, encoded in 4 bytes and decoded again (decodeFrame), so that the binary walk (this array)
    // and the wide walk (the code alone) use the same float32 frame; half extents measured in exactly that frame, inflated so
    // that rounding can never cut a triangle off. o = {centre u, v, n, he u | u, he v | v, he n | n, frame code}. Nodes whose
    // normals disagree keep only their axis-aligned box.
    __global__ void __launch_bounds__(256) meshObbKernel(const MeshBuildIn M, const BvhNode* __restrict__ nodes, const uint32_t* __restrict__ nodeBegin,
                                                         const uint32_t* __restrict__ nodeEnd, const uint32_t* __restrict__ order, uint32_t nNodes,
                                                         double inflate, float* __restrict__ obb)
    {
        const uint32_t node = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31u;
        if (node >= nNodes) return;
        float* o = obb + 16 * (size_t)node;
        if (lane < 16u) o[lane] = (lane == 3u || lane == 7u || lane == 11u) ? 3.402823466e+38f : 0.0f;
        __syncwarp();
        const uint32_t b = nodeBegin[node], e = nodeEnd[node];
        if (e - b > 32768u) return;
        double N[3] = { 0, 0, 0 }, total = 0.0;
        for (uint32_t k = b + lane; k < e; k += 32u)
        {
            const uint32_t t = order[k];
            const F3 a = vertOf(M, t, 0), bb = vertOf(M, t, 1), c = vertOf(M, t, 2);
            const double e1[3] = { (double)bb.x - a.x, (double)bb.y - a.y, (double)bb.z - a.z }, e2[3] = { (double)c.x - a.x, (double)c.y - a.y, (double)c.z - a.z };
            const double cr[3] = { e1[1] * e2[2] - e1[2] * e2[1], e1[2] * e2[0] - e1[0] * e2[2], e1[0] * e2[1] - e1[1] * e2[0] };
            N[0] += cr[0]; N[1] += cr[1]; N[2] += cr[2];
            total += sqrt(cr[0] * cr[0] + cr[1] * cr[1] + cr[2] * cr[2]);
        }
        #pragma unroll
        for (int s = 16; s > 0; s >>= 1)
        {
            N[0] += __shfl_xor_sync(0xFFFFFFFFu, N[0], s); N[1] += __shfl_xor_sync(0xFFFFFFFFu, N[1], s); N[2] += __shfl_xor_sync(0xFFFFFFFFu, N[2], s);
            total += __shfl_xor_sync(0xFFFFFFFFu, total, s);
        }
        const double len = sqrt(N[0] * N[0] + N[1] * N[1] + N[2] * N[2]);
        if (!(len > 0.5 * total) || !(len > 0.0)) return;
        const double nn[3] = { N[0] / len, N[1] / len, N[2] / len };
        int ax = 0;                                              // tangents: the coordinate axis least aligned with n, made orthogonal
        if (fabs(nn[1]) < fabs(nn[ax])) ax = 1;
        if (fabs(nn[2]) < fabs(nn[ax])) ax = 2;
        double u[3] = { -nn[ax] * nn[0], -nn[ax] * nn[1], -nn[ax] * nn[2] };
        u[ax] += 1.0;
        const double ul = sqrt(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
        for (int d = 0; d < 3; ++d) u[d] /= ul;
        const double frame[3][3] = { { u[0], u[1], u[2] },
                                     { nn[1] * u[2] - nn[2] * u[1], nn[2] * u[0] - nn[0] * u[2], nn[0] * u[1] - nn[1] * u[0] },
                                     { nn[0], nn[1], nn[2] } };
        // the frame the walks use is the one decoded from its 4-byte code (mesh_eval.cuh), and the extents are measured in it
        const uint32_t code = encodeFrame(frame);
        F3 du, dw, dn;
        decodeFrame(code, du, dw, dn);
        const float fu[3] = { du.x, du.y, du.z }, fw[3] = { dw.x, dw.y, dw.z }, fn[3] = { dn.x, dn.y, dn.z };
        double lo[3] = { 1e300, 1e300, 1e300 }, hi[3] = { -1e300, -1e300, -1e300 };
        for (uint32_t k = b + lane; k < e; k += 32u)
        {
            const uint32_t t = order[k];
            for (uint32_t c = 0; c < 3; ++c)
            {
                const F3 p = vertOf(M, t, c);
                const double q[3] = { (double)p.x * fu[0] + (double)p.y * fu[1] + (double)p.z * fu[2],
                                      (double)p.x * fw[0] + (double)p.y * fw[1] + (double)p.z * fw[2],
                                      (double)p.x * fn[0] + (double)p.y * fn[1] + (double)p.z * fn[2] };
                for (int d = 0; d < 3; ++d) { lo[d] = fmin(lo[d], q[d]); hi[d] = fmax(hi[d], q[d]); }
            }
        }
        #pragma unroll
        for (int s = 16; s > 0; s >>= 1)
            for (int d = 0; d < 3; ++d)
            {
                lo[d] = fmin(lo[d], __shfl_xor_sync(0xFFFFFFFFu, lo[d], s));
                hi[d] = fmax(hi[d], __shfl_xor_sync(0xFFFFFFFFu, hi[d], s));
            }
        if (lane == 0u)
        {
            // centre in frame coordinates (the traversal projects p onto the axes and subtracts these)
            o[0] = (float)(0.5 * (lo[0] + hi[0])); o[1] = (float)(0.5 * (lo[1] + hi[1])); o[2] = (float)(0.5 * (lo[2] + hi[2]));
            for (int d = 0; d < 3; ++d)
            {
                const double c = (double)o[d];
                const double he = fmax(hi[d] - c, c - lo[d]) + inflate;
                o[3 + 4 * d] = nextafterf((float)he, 3.402823466e+38f);
            }
            o[4] = fu[0]; o[5] = fu[1]; o[6] = fu[2];
            o[8] = fw[0]; o[9] = fw[1]; o[10] = fw[2];
            o[12] = fn[0]; o[13] = fn[1]; o[14] = fn[2]; o[15] = __uint_as_float(code);
        }
    }

    // node -> triangle range, and which nodes root a 4-wide node (internal nodes at even depth)
    __global__ void __launch_bounds__(256) meshNodeRangesKernel(const BvhNode* __restrict__ nodes, const uint32_t* __restrict__ parent,
                                                                const uint32_t* __restrict__ nodeDepth, uint32_t nNodes, uint32_t nTris,
                                                                uint32_t* __restrict__ nodeBegin, uint32_t* __restrict__ nodeEnd, uint32_t* __restrict__ wideFlag)
    {
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= nNodes) return;
        // leftmost / rightmost leaf below node i
        uint32_t l = i, r = i;
        while (!(nodes[l].b & 0x80000000u)) l = nodes[l].a;
        while (!(nodes[r].b & 0x80000000u)) r = nodes[r].b;
        nodeBegin[i] = nodes[l].a;
        nodeEnd[i] = nodes[r].a + (nodes[r].b & 0x7FFFFFFFu);
        wideFlag[i] = (!(nodes[i].b & 0x80000000u) && (nodeDepth[i] & 1u) == 0u) ? 1u : 0u;
    }

    // 4-wide collapse for meshSampleKernel: a wide node holds the grandchildren of a binary node (or its children where they are
    // leaves) in one 128-byte record, one float4 per field with child k in component k:
    //   { child reference (kNoNode | leaf: 0x80000000 | count << 28 | first slot | wide index) }, { frame code (decodeFrame) },
    //   { centre u }, { centre v }, { centre n }, { half extent u }, { half extent v }, { half extent n }.
    // Nodes without an oriented box get their axis-aligned box with the identity frame code.
    constexpr int kWideFloats = 32;
    __device__ __forceinline__ void putWideChild(float* __restrict__ out, int k, uint32_t ref, uint32_t code, const float* centre, const float* he)
    {
        out[k] = __uint_as_float(ref);
        out[4 + k] = __uint_as_float(code);
        for (int d = 0; d < 3; ++d) { out[8 + 4 * d + k] = centre[d]; out[20 + 4 * d + k] = he[d]; }
    }
    __device__ __forceinline__ void putAbsentChild(float* __restrict__ out, int k)
    {
        const float zero[3] = { 0.0f, 0.0f, 0.0f }, never[3] = { -3.0e38f, -3.0e38f, -3.0e38f };     // |q| - he overflows to +inf
        putWideChild(out, k, 0xFFFFFFFFu, kIdentityFrame, zero, never);
    }

    __global__ void __launch_bounds__(256) meshWideKernel(const BvhNode* __restrict__ nodes, const float* __restrict__ obb, const uint32_t* __restrict__ wideFlag,
                                                          const uint32_t* __restrict__ wideIdx, uint32_t nNodes, double inflate, float* __restrict__ wide)
    {
        const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
        if (b >= nNodes || !wideFlag[b]) return;
        float* out = wide + kWideFloats * (size_t)wideIdx[b];
        uint32_t kids[4], nk = 0;
        const uint32_t two[2] = { nodes[b].a, nodes[b].b };
        for (int s = 0; s < 2; ++s)
        {
            const BvhNode c = nodes[two[s]];
            if (c.b & 0x80000000u) kids[nk++] = two[s];
            else { kids[nk++] = c.a; kids[nk++] = c.b; }
        }
        for (uint32_t k = 0; k < 4; ++k)
        {
            if (k >= nk) { putAbsentChild(out, k); continue; }
            const BvhNode c = nodes[kids[k]];
            const float* o = obb + 16 * (size_t)kids[k];
            const uint32_t ref = (c.b & 0x80000000u) ? (0x80000000u | ((c.b & 7u) << 28) | c.a) : wideIdx[kids[k]];
            if (o[3] < 1e38f)
            {
                const float centre[3] = { o[0], o[1], o[2] }, he[3] = { o[3], o[7], o[11] };
                putWideChild(out, k, ref, __float_as_uint(o[15]), centre, he);
            }
            else
            {
                float centre[3], he[3];
                for (int d = 0; d < 3; ++d)
                {
                    const double lo = c.mn[d], hi = c.mx[d];
                    centre[d] = (float)(0.5 * (lo + hi));
                    const double ce = (double)centre[d];
                    he[d] = nextafterf((float)(fmax(hi - ce, ce - lo) + inflate), 3.402823466e+38f);
                }
                putWideChild(out, k, ref, kIdentityFrame, centre, he);        // u = x, v = y, n = z
            }
        }
    }

    // a mesh of at most 4 triangles is one leaf: the wide tree is a root with that single child, whose box contains everything
    __global__ void meshWideSingleLeafKernel(const BvhNode* __restrict__ nodes, float* __restrict__ wide)
    {
        if (threadIdx.x != 0 || blockIdx.x != 0) return;
        const float zero[3] = { 0.0f, 0.0f, 0.0f }, all[3] = { 3.0e38f, 3.0e38f, 3.0e38f };
        putWideChild(wide, 0, 0x80000000u | ((nodes[0].b & 7u) << 28) | nodes[0].a, kIdentityFrame, zero, all);
        for (int k = 1; k < 4; ++k) putAbsentChild(wide, k);
    }

    // triangle vertices in BVH order: 3 float4 per slot, the original triangle index rides in a.w
    __global__ void __launch_bounds__(256) meshSlotsKernel(const MeshBuildIn M, const uint32_t* __restrict__ order, float4* __restrict__ tv)
    {
        const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
        if (slot >= M.nTris) return;
        const uint32_t t = order[slot];
        const F3 a = vertOf(M, t, 0), b = vertOf(M, t, 1), c = vertOf(M, t, 2);
        tv[3 * (size_t)slot] = make_float4(a.x, a.y, a.z, __uint_as_float(t));
        tv[3 * (size_t)slot + 1] = make_float4(b.x, b.y, b.z, 0.0f);
        tv[3 * (size_t)slot + 2] = make_float4(c.x, c.y, c.z, 0.0f);
    }

    __global__ void fillU32Kernel(uint32_t* __restrict__ p, size_t n, uint32_t v)
    {
        const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i < n) p[i] = v;
    }
}
