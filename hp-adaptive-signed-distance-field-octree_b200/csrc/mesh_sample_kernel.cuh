// mesh_sample_kernel.cuh — F at the Gauss-Legendre points of a chunk of fits when the SDF program is a single triangle
// mesh: the kernel that dominates every mesh build (configs 3-5 of BASELINE.json).
//
// What ncu said about calling the per-thread traversal (mesh_eval.cuh) from sampleKernel, one sample per thread:
// 5.9 of 32 lanes active per issued instruction. A closest-triangle query alternates between ~80-instruction node steps
// and ~170-instruction exact triangle tests (ClosestSimplexToPt mirrored operation by operation), the lanes of a warp need
// different numbers of node steps to reach their next leaf (the node loop ran 788 iterations per warp for 111 per lane),
// and a lane whose query is finished idles until the slowest one of its warp is.
//
// Here the warp is a scheduler over 32 independent query state machines:
//   * every loop iteration is EITHER a node step OR a triangle test for all lanes that have one pending — the choice is
//     warp-uniform (ballots), so the two instruction streams are never serialised against each other;
//   * reaching a leaf does not test it: the leaf goes into a 4-entry per-lane queue and the lane keeps walking; triangle
//     iterations run when at least `triThreshold` (12) lanes have a triangle waiting (or nobody has a node left), re-checking the leaf's
//     bound against the lane's current best first;
//   * a lane that finishes its query writes the sample and takes the next one (warps grab 32-128 samples at a time from a
//     global counter), so lanes do not wait for their neighbours and far / near cells balance across the grid;
//   * the tree is walked in its 4-wide collapse (mesh_build.cuh: meshWideKernel), one 128-byte record (one cache line: four
//     child references, four 4-byte frame codes, four oriented boxes in f32) per node step, read as 8 float4; the frames are
//     decoded in registers (mesh_eval.cuh: decodeFrame). The walk is bound by L1 throughput and latency, and leaf sizes
//     1 / 2 / 4 / 7 measured 98 / 90 / 83 / 80 ms — node steps are the cost;
//   * a stack entry is (node, bound) in 8 bytes: one local-memory access per push or pop;
//   * when the samples run out, lanes without work take sub-trees from lanes that still have a stack (tail phase below);
// Results are those of meshSignedDistanceF: same exact test, same (smallest f32 d2, lowest triangle index) winner, same
// conservative pruning — the order in which candidates are met does not matter to that rule.
#pragma once
#include "hp_common.h"
#include "mesh_eval.cuh"

namespace hpsdf
{
    constexpr int      kMeshQueue = 4;
    constexpr int      kMeshStack = 48;         // >= 3 pushes x 14 levels: the 4-wide tree of the largest accepted mesh (2^28 triangles, median split)
    constexpr uint32_t kNoNode    = 0xFFFFFFFFu;

    __device__ __forceinline__ unsigned long long stackEntry(uint32_t node, float bound)
    {
        return (unsigned long long)node | ((unsigned long long)__float_as_uint(bound) << 32);
    }

    __global__ void __launch_bounds__(256, 4)
    meshSampleKernel(const FitTask* __restrict__ tasks, unsigned long long nSamples, int D, const DeviceMeshView* __restrict__ mesh,
                     const RootMap map, const FitTablesDev tab, double* __restrict__ samples, unsigned long long* __restrict__ counter,
                     const unsigned grab, const int triThreshold,   // (triThreshold: see launchOne)
                     const int handOver,                            // 1 = tail phase on (0: diagnostics, HPSDF_MESH_NO_HANDOVER)
                     unsigned long long* __restrict__ stats)        // diagnostics (HPSDF_MESH_STATS): histogram of node steps per query, or nullptr
    {
        const float4* __restrict__ wide = (const float4*)mesh->wide;           // 8 float4 per 4-wide node (meshWideKernel)
        const float4* __restrict__ tv = (const float4*)mesh->triVerts;
        const double* __restrict__ roots = tab.roots[D];
        const unsigned n = (unsigned)fitRule(D), n2 = n * n, n3 = n2 * n;
        const unsigned lane = threadIdx.x & 31u, ltMask = (1u << lane) - 1u;

        // per-lane query state
        long long sid = -1;                       // sample index, -1 = idle
        F3 p = f3(0.0f, 0.0f, 0.0f);
        MeshHit h;
        unsigned long long stack[kMeshStack];             // node | bound bits << 32
        int sp = 0;
        uint32_t cur = kNoNode; float curD = 0.0f;       // wide node (or leaf reference, bit 31) to process and its bound
        uint32_t qLeaf[kMeshQueue]; float qD[kMeshQueue];        // circular: head qh, count qn; entry = leaf reference
        int qh = 0, qn = 0;
        unsigned steps = 0;                                      // node steps of the lane's current query
        // warp-uniform work cursor
        unsigned long long cursor = 0, grabEnd = 0;
        bool exhausted = false;

        // One entry per call: a stale entry (its bound no longer beats the lane's best) is recognised by the next node step,
        // which then pops again — a divergent "skip the stale ones" loop here ran with 2-4 active lanes and drew 29 % of the
        // kernel's stall samples on its dependent local-memory loads.
        auto pop = [&]()
        {
            if (sp > 0) { --sp; const unsigned long long e = stack[sp]; cur = (uint32_t)e; curD = __uint_as_float((uint32_t)(e >> 32)); }
            else cur = kNoNode;
        };

        // One step for every lane that has one: a node step or a triangle test, chosen warp-uniformly. `active`: the lane works
        // on a query (its own sample, or in the tail phase a sub-tree of somebody else's); `bound`: the squared distance nothing
        // farther than which can win (the lane's own best; in the tail phase the best of all lanes working on the same sample).
        auto step = [&](const bool active, const float bound)
        {
            const bool wantNode = active && cur != kNoNode && qn < kMeshQueue;
            const unsigned nodeMask = __ballot_sync(0xFFFFFFFFu, wantNode);
            const unsigned triMask = __ballot_sync(0xFFFFFFFFu, qn > 0);
            if (nodeMask != 0u && __popc(triMask) < triThreshold)
            {
                if (wantNode)
                {
                    ++steps;
                    if (curD > bound * 1.000001f) pop();                         // went stale on the stack
                    else if (cur & 0x80000000u)
                    {
                        const int slot = (qh + qn) & (kMeshQueue - 1);
                        qLeaf[slot] = cur;                                       // 0x80000000 | count << 28 | first triangle slot
                        qD[slot] = curD;
                        ++qn;
                        pop();
                    }
                    else
                    {
                        // one cache line per step: the four child references, frame codes and boxes of the node, all requested at once
                        const float4* __restrict__ w = wide + 8 * (size_t)cur;
                        const float4 hdr = __ldg(w), code = __ldg(w + 1), cu = __ldg(w + 2), cv = __ldg(w + 3), cn = __ldg(w + 4),
                                     hu = __ldg(w + 5), hv = __ldg(w + 6), hn = __ldg(w + 7);
                        const uint32_t ref[4] = { __float_as_uint(hdr.x), __float_as_uint(hdr.y), __float_as_uint(hdr.z), __float_as_uint(hdr.w) };
                        const float lim = bound * 1.000001f;
                        float cd[4];
                        #pragma unroll
                        for (int k = 0; k < 4; ++k)
                        {
                            const auto at = [k](const float4& q) { return k == 0 ? q.x : k == 1 ? q.y : k == 2 ? q.z : q.w; };
                            F3 u, v, nrm;
                            decodeFrame(__float_as_uint(at(code)), u, v, nrm);
                            const float d = obbDist2(make_float4(at(cu), at(cv), at(cn), at(hu)), make_float4(u.x, u.y, u.z, at(hv)),
                                                     make_float4(v.x, v.y, v.z, at(hn)), make_float4(nrm.x, nrm.y, nrm.z, 0.0f), p);
                            cd[k] = (ref[k] != kNoNode && d <= lim) ? d : 3.402823466e+38f;          // FLT_MAX = "do not visit" (lim < FLT_MAX once a triangle was seen; before that every real child passes)
                        }
                        // visit order: nearest first; the others go on the stack farthest first so that the nearest of them is popped next
                        uint32_t r0 = ref[0], r1 = ref[1], r2 = ref[2], r3 = ref[3];
                        float d0 = cd[0], d1 = cd[1], d2 = cd[2], d3 = cd[3];
                        #define HPSDF_CSWAP(da, ra, db, rb) if (db < da) { const float td = da; da = db; db = td; const uint32_t tr = ra; ra = rb; rb = tr; }
                        HPSDF_CSWAP(d0, r0, d1, r1) HPSDF_CSWAP(d2, r2, d3, r3) HPSDF_CSWAP(d0, r0, d2, r2) HPSDF_CSWAP(d1, r1, d3, r3) HPSDF_CSWAP(d1, r1, d2, r2)
                        #undef HPSDF_CSWAP
                        const bool v0 = d0 < 3.0e38f;
                        if (d3 < 3.0e38f && sp < kMeshStack) stack[sp++] = stackEntry(r3, d3);
                        if (d2 < 3.0e38f && sp < kMeshStack) stack[sp++] = stackEntry(r2, d2);
                        if (d1 < 3.0e38f && sp < kMeshStack) stack[sp++] = stackEntry(r1, d1);
                        if (v0) { cur = r0; curD = d0; }
                        else pop();
                    }
                }
            }
            else if (qn > 0)
            {
                const uint32_t e = qLeaf[qh];
                const uint32_t first = e & 0x0FFFFFFFu, cnt = (e >> 28) & 7u;
                if (qD[qh] <= bound * 1.000001f)                               // else: pruned while it waited
                {
                    // the whole leaf in one iteration (3-4 triangles): the scheduler's ballots are paid once per leaf
                    #pragma unroll 1
                    for (uint32_t t = 0; t < cnt; ++t)
                    {
                        const float4 A = __ldg(tv + 3 * (size_t)(first + t)), B = __ldg(tv + 3 * (size_t)(first + t) + 1), C = __ldg(tv + 3 * (size_t)(first + t) + 2);
                        const uint32_t tri = __float_as_uint(A.w);
                        int s, id;
                        const F3 cp = closestSimplex(p, f3(A.x, A.y, A.z), f3(B.x, B.y, B.z), f3(C.x, C.y, C.z), s, id);
                        const F3 d = sub3(p, cp);
                        const float d2 = dot3(d, d);                           // (pt - closestPt).squaredNorm(), BVH.cpp:320
                        if (d2 < h.best || (d2 == h.best && tri < h.tri)) { h.best = d2; h.tri = tri; h.simplex = s; h.id = id; h.pt = cp; }
                    }
                }
                qh = (qh + 1) & (kMeshQueue - 1);
                --qn;
            }
        };

        auto retire = [&]()
        {
            samples[sid] = (double)finishHit(mesh, p, h);
            sid = -1;
            if (stats)
            {
                atomicAdd(stats + (steps ? 32 - __clz(steps) : 0), 1ull);      // bucket b: steps in [2^(b-1), 2^b)
                atomicAdd(stats + 40, (unsigned long long)steps);
                atomicMax(stats + 41, (unsigned long long)steps);
            }
        };

        // ==== main phase: every lane owns a query; finished lanes take the next sample ==================================================
        for (;;)
        {
            // ---- retire finished queries, hand out new samples -----------------------------------------------------
            if (sid >= 0 && cur == kNoNode && qn == 0) retire();
            unsigned idle = __ballot_sync(0xFFFFFFFFu, sid < 0);
            while (idle && !exhausted)
            {
                if (cursor == grabEnd)
                {
                    unsigned long long g = 0;
                    if (lane == 0) g = atomicAdd(counter, (unsigned long long)grab);
                    g = __shfl_sync(0xFFFFFFFFu, g, 0);
                    if (g >= nSamples) { exhausted = true; break; }
                    cursor = g;
                    grabEnd = g + grab < nSamples ? g + grab : nSamples;
                }
                const unsigned avail = (unsigned)(grabEnd - cursor), want = (unsigned)__popc(idle);
                const unsigned rank = (unsigned)__popc(idle & ltMask);
                if (sid < 0 && rank < avail)
                {
                    sid = (long long)(cursor + rank);
                    const unsigned long long g = (unsigned long long)sid;
                    const unsigned fit = (unsigned)(g / n3), s = (unsigned)(g - (unsigned long long)fit * n3);
                    const unsigned k = s / n2, col = s - k * n2, j = col / n, i = col - j * n;
                    const float4 cell = *reinterpret_cast<const float4*>(&tasks[fit]);          // cx, cy, cz, half
                    const double half = (double)cell.w;
                    // the same expressions as the closed-form fit kernels (samplePos), then the float32 cast of the mesh SDF glue
                    p = f3((float)samplePos(roots[i], half, (double)cell.x, map.sizes[0], map.centre[0]),
                           (float)samplePos(roots[j], half, (double)cell.y, map.sizes[1], map.centre[1]),
                           (float)samplePos(roots[k], half, (double)cell.z, map.sizes[2], map.centre[2]));
                    h = MeshHit();
                    h.pt = p;
                    sp = 0; cur = 0; curD = 0.0f; qh = 0; qn = 0; steps = 0;
                }
                cursor += want < avail ? want : avail;
                idle = __ballot_sync(0xFFFFFFFFu, sid < 0);
            }
            if (idle == 0xFFFFFFFFu) return;                                  // nothing in flight and nothing left to take
            if (idle && handOver) break;                                      // no samples left and some lanes have nothing to do: tail phase
            step(true, h.best);
        }

        // ==== tail phase: lanes without work take sub-trees from lanes that have some ======================================================
        // The end of a launch used to be a few lanes finishing 300-600-step queries (points near the medial axis, which is where
        // hp-refinement concentrates) while the rest of the warp had run out of samples: a small launch lasted as long as its
        // slowest query, 0.5-0.9 ms. Here a lane without work takes the top stack entry (a whole sub-tree) of a lane that has one,
        // walks it against the best distance of everybody working on that sample (shared memory, atomicMin on the float bits:
        // d2 >= 0, so integer order = float order), and hands its best hit back when it runs dry; helpers can be robbed in turn.
        // (smallest d2, lowest triangle index) is a total order and every lane prunes against a bound that is no better than the
        // final one, so the winner is the same triangle as before.
        __shared__ unsigned sBest[8][32];
        unsigned* wBest = sBest[threadIdx.x >> 5];
        int owner = -1;                                          // >= 0: this lane walks a sub-tree handed over by that lane (sid < 0 then)
        int root = (int)lane;                                    // the lane whose sample the sub-tree belongs to (chains: the first donor)
        int helpers = 0;                                         // sub-trees handed over by this lane and not merged back yet
        int handedOver = 0;                                      // warp-uniform: the same, for the whole warp
        wBest[lane] = 0x7F7FFFFFu;                               // FLT_MAX
        __syncwarp();
        for (;;)
        {
            if (handedOver)
            {
                // helpers that ran dry give their best hit to the lane they took the sub-tree from
                unsigned fin = __ballot_sync(0xFFFFFFFFu, owner >= 0 && cur == kNoNode && qn == 0 && helpers == 0);
                while (fin)
                {
                    const int l = __ffs(fin) - 1;
                    fin &= fin - 1u;
                    const int own = __shfl_sync(0xFFFFFFFFu, owner, l);
                    const float hb = __shfl_sync(0xFFFFFFFFu, h.best, l);
                    const uint32_t ht = __shfl_sync(0xFFFFFFFFu, h.tri, l);
                    const int hs = __shfl_sync(0xFFFFFFFFu, h.simplex, l), hi = __shfl_sync(0xFFFFFFFFu, h.id, l);
                    const float hx = __shfl_sync(0xFFFFFFFFu, h.pt.x, l), hy = __shfl_sync(0xFFFFFFFFu, h.pt.y, l), hz = __shfl_sync(0xFFFFFFFFu, h.pt.z, l);
                    if ((int)lane == own)
                    {
                        if (hb < h.best || (hb == h.best && ht < h.tri)) { h.best = hb; h.tri = ht; h.simplex = hs; h.id = hi; h.pt = f3(hx, hy, hz); }
                        --helpers;
                    }
                    if ((int)lane == l) owner = -1;
                    --handedOver;
                }
            }
            if (sid >= 0 && cur == kNoNode && qn == 0 && helpers == 0) retire();
            const unsigned idle = __ballot_sync(0xFFFFFFFFu, sid < 0 && owner < 0);
            if (idle == 0xFFFFFFFFu) return;
            if (idle)
            {
                // the i-th lane without work takes the top stack entry of the i-th lane that has one to spare (only from lanes that
                // have seen a triangle: before that nothing can be pruned and a helper would walk its whole sub-tree)
                const bool canGive = (sid >= 0 || owner >= 0) && sp > 0 && cur != kNoNode && h.best < 3.0e38f;
                const unsigned donors = __ballot_sync(0xFFFFFFFFu, canGive);
                if (donors)
                {
                    const int nPairs = min(__popc(idle), __popc(donors));
                    const bool take = sid < 0 && owner < 0 && (int)__popc(idle & ltMask) < nPairs;
                    const bool give = canGive && (int)__popc(donors & ltMask) < nPairs;
                    const int src = take ? (int)__fns(donors, 0u, __popc(idle & ltMask) + 1) : (int)lane;
                    uint32_t gN = kNoNode; float gD = 0.0f;
                    if (give) { --sp; const unsigned long long e = stack[sp]; gN = (uint32_t)e; gD = __uint_as_float((uint32_t)(e >> 32)); ++helpers; }
                    const uint32_t tN = __shfl_sync(0xFFFFFFFFu, gN, src);
                    const float tD = __shfl_sync(0xFFFFFFFFu, gD, src);
                    const int tRoot = __shfl_sync(0xFFFFFFFFu, root, src);
                    const float px = __shfl_sync(0xFFFFFFFFu, p.x, src), py = __shfl_sync(0xFFFFFFFFu, p.y, src), pz = __shfl_sync(0xFFFFFFFFu, p.z, src);
                    const float hb = __shfl_sync(0xFFFFFFFFu, h.best, src);
                    const uint32_t ht = __shfl_sync(0xFFFFFFFFu, h.tri, src);
                    const int hs = __shfl_sync(0xFFFFFFFFu, h.simplex, src), hi = __shfl_sync(0xFFFFFFFFu, h.id, src);
                    const float hx = __shfl_sync(0xFFFFFFFFu, h.pt.x, src), hy = __shfl_sync(0xFFFFFFFFu, h.pt.y, src), hz = __shfl_sync(0xFFFFFFFFu, h.pt.z, src);
                    if (take)
                    {
                        owner = src; root = tRoot;
                        p = f3(px, py, pz);
                        h.best = hb; h.tri = ht; h.simplex = hs; h.id = hi; h.pt = f3(hx, hy, hz);
                        cur = tN; curD = tD; sp = 0; qh = 0; qn = 0; helpers = 0;
                    }
                    handedOver += nPairs;
                }
            }
            const bool active = sid >= 0 || owner >= 0;
            if (active) atomicMin(wBest + root, __float_as_uint(h.best));
            __syncwarp();
            step(active, active ? __uint_as_float(wBest[root]) : 0.0f);
        }
    }
}
