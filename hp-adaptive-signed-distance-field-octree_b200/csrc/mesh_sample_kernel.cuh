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
//   * reaching a leaf does not test it: a node step puts the leaf children that pass the bound straight into an 8-entry
//     per-lane queue (nearest first, in shared memory) and the lane keeps walking; only inner children become the next node
//     or go on the stack, so every node step that is not a stale pop reads a node. Triangle iterations run when at least
//     `triThreshold` (16) lanes have a triangle waiting (or nobody has a node left), re-checking the leaf's bound against the
//     lane's current best first;
//   * a lane that finishes its query writes the sample and takes the next one (warps grab 32-128 samples at a time from a
//     global counter), so lanes do not wait for their neighbours and far / near cells balance across the grid;
//   * the tree is walked in its 4-wide collapse (mesh_build.cuh: meshWideKernel), one 128-byte record (one cache line: four
//     child references, four 4-byte frame codes, four oriented boxes in f32) per node step, read as 8 float4; the frames are
//     decoded in registers (mesh_eval.cuh: decodeFrame). The walk is bound by L1 throughput and latency, and leaf sizes
//     1 / 2 / 4 / 7 measured 98 / 90 / 83 / 80 ms — node steps are the cost;
//   * a stack entry is (node, bound) in 8 bytes: one local-memory access per push or pop; it also records how many entries
//     below it came from the same node step. Those are its farther siblings, so once its bound is stale theirs are too, and
//     a stale pop drops them without a step of their own;
//   * when the samples run out, lanes without work take sub-trees from lanes that still have a stack (tail phase below);
//   * a query does not start at the root: meshCutKernel (below) first cuts the top of the tree once per fit, and every sample of
//     the fit starts at that cut with a pruning bound from the distance at the fit's centre (DESIGN §7);
// Results are those of meshSignedDistanceF: same exact test, same (smallest f32 d2, lowest triangle index) winner, same
// conservative pruning — the order in which candidates are met does not matter to that rule.
#pragma once
#include "hp_common.h"
#include "mesh_eval.cuh"

namespace hpsdf
{
    constexpr int      kMeshQueue = 8;          // a node step needs room for 4 leaves, so up to 4 earlier ones can wait and the queue never overflows (power of 2: ring index)
    constexpr int      kMeshStack = 48;         // >= 3 pushes x 14 levels: the 4-wide tree of the largest accepted mesh (2^28 triangles, median split)
    constexpr uint32_t kNoNode    = 0xFFFFFFFFu;
    // A stack entry and `cur` hold the wide-node index in bits 0-27 and, in bits 28-29, how many entries directly below it on
    // the stack were pushed by the same node step (0-3). Bit 30 marks a record of the cut buffer instead of a wide node. Those
    // bits are free: the builder rejects meshes with 2^28 or more wide nodes (mesh.cpp), a launch has fewer than 2^28 cut
    // records (launchOne), and leaf references (bit 31) go to the leaf queue, never on the stack.
    constexpr uint32_t kNodeIndexMask = 0x0FFFFFFFu;
    constexpr int      kGroupShift    = 28;
    constexpr uint32_t kCutBit        = 0x40000000u;

    // The cut of a fit (meshCutKernel): up to kMeshCut child entries of the 4-wide tree that together hold every triangle that
    // can be the closest one of any sample of the fit, written as 128-byte records in exactly the wide-node format, 4 entries
    // each. A fit owns kCutStride records of the buffer: a header { c.x, c.y, c.z, dc } { record count, 0, 0, 0 } (c: centre
    // of the fit's sample box, dc: bound of the distance at c, rounded up) and then its cut records, nearest entries first.
    // At most 16 entries: on C3, with an exact centre distance instead of the greedy one, 8 / 16 / 32 gave 44.8 / 43.6 / 42.3 node visits per query and 49.4 / 48.6 / 48.3 ms per
    // step (profiles/r5_mesh_cut.md); beyond 16 the cut records could take the stack past kMeshStack on the deepest meshes.
    constexpr int      kMeshCut     = 16;
    constexpr int      kCutRecords  = (kMeshCut + 3) / 4;
    constexpr int      kCutStride   = kCutRecords + 1;
    // cut buffer per sample double of the scratch: a fit has at least 5^3 samples (fitRule(1))
    constexpr size_t   kCutSamplesPerFit = 125;
    static_assert(kCutRecords <= 4, "the header holds the stack bounds of 3 records after the first, and a group count is 2 bits");
    // HPSDF_MESH_STATS: per-thread event counters in dynamic shared memory, [counter][threadIdx], added to words 42.. of
    // the stats buffer when the block ends (fit_kernels.cuh: printMeshStats)
    enum MeshStat { kStatNodeVisit, kStatStalePop, kStatGroupDrop, kStatLeafTest, kStatLeafPruned, kStatWarpNodeIter, kStatWarpTriIter, kMeshStatCount };
    constexpr int kMeshStatWord = 42;

    __device__ __forceinline__ unsigned long long stackEntry(uint32_t node, float bound)
    {
        return (unsigned long long)node | ((unsigned long long)__float_as_uint(bound) << 32);
    }

    // HPSDF_MESH_STATS words of meshCutKernel: entries summed over fits, largest cut, fits whose cut expanded no node below the
    // root, fits
    constexpr int kCutStatWord = 56;

    // One warp per fit: the cut of the 4-wide tree that every sample of the fit starts from (meshSampleKernel), and the bound
    // that seeds their pruning. Exactness (DESIGN §7): with c the centre of the fit's f32 sample box and r its half-diagonal,
    // and dc the distance from c to some triangle T, every sample x has d(x) <= d(x, T) <= dc + |x - c| <= U = dc + r, so a
    // child whose box is farther than U from every sample
    // (dist(c, box) - r > U) holds no triangle that can win or tie at any sample of the fit. All bounds carry a relative 1e-5
    // and an absolute 1e-5 of the mesh size (mesh->inflate) against f32 rounding, and the box distances are computed in
    // double from the f32 frame and extents of the record, shrunk by 2e-6 (the decoded frame stretches by <= 1.6 * 2^-24).
    __global__ void __launch_bounds__(128)
    meshCutKernel(const FitTask* __restrict__ tasks, unsigned nFits, int D, const DeviceMeshView* __restrict__ mesh, const RootMap map,
                  const FitTablesDev tab, float4* __restrict__ cut, unsigned long long* __restrict__ stats)
    {
        __shared__ uint32_t sEnt[4][kMeshCut][8];       // per warp: the cut's entries (child reference, frame code, centre, half extents)
        __shared__ float    sLb[4][kMeshCut];            // lower bound of the distance from c, for the order of expansion and output
        __shared__ uint8_t  sFrozen[4][kMeshCut];        // 1: expanding this entry would overflow the cut
        __shared__ uint8_t  sOrd[4][kMeshCut];
        const unsigned wib = threadIdx.x >> 5, lane = threadIdx.x & 31u;
        const unsigned fit = blockIdx.x * 4u + wib;
        if (fit >= nFits) return;                        // warp-uniform
        uint32_t (*ent)[8] = sEnt[wib];
        float* lbs = sLb[wib];
        uint8_t* frozen = sFrozen[wib];
        const float4* __restrict__ wide = (const float4*)mesh->wide;

        // the f32 box of the sample positions: the same samplePos expressions and cast as meshSampleKernel, over every root
        const unsigned n = (unsigned)fitRule(D);
        const double* __restrict__ roots = tab.roots[D];
        const float4 cell = *reinterpret_cast<const float4*>(&tasks[fit]);          // cx, cy, cz, half
        const double cc[3] = { (double)cell.x, (double)cell.y, (double)cell.z };
        float lo[3], hi[3];
        #pragma unroll
        for (int d = 0; d < 3; ++d)
        {
            lo[d] = 3.402823466e+38f; hi[d] = -3.402823466e+38f;
            for (unsigned i = lane; i < n; i += 32u)
            {
                const float x = (float)samplePos(roots[i], (double)cell.w, cc[d], map.sizes[d], map.centre[d]);
                lo[d] = fminf(lo[d], x); hi[d] = fmaxf(hi[d], x);
            }
            #pragma unroll
            for (int s = 16; s > 0; s >>= 1)
            {
                lo[d] = fminf(lo[d], __shfl_xor_sync(0xFFFFFFFFu, lo[d], s));
                hi[d] = fmaxf(hi[d], __shfl_xor_sync(0xFFFFFFFFu, hi[d], s));
            }
        }
        const F3 c = f3((float)(0.5 * ((double)lo[0] + hi[0])), (float)(0.5 * ((double)lo[1] + hi[1])), (float)(0.5 * ((double)lo[2] + hi[2])));
        const double cd[3] = { (double)c.x, (double)c.y, (double)c.z };
        double r2 = 0.0;
        #pragma unroll
        for (int d = 0; d < 3; ++d) { const double e = fmax(cd[d] - lo[d], hi[d] - cd[d]); r2 += e * e; }
        const double r = sqrt(r2) * (1.0 + 1e-5);
        const double eps = (double)mesh->inflate;

        // dc: the distance from c to the closest triangle of the leaf reached by always stepping to the child whose box is
        // nearest to c. It bounds d(c) from above like the exact closest triangle would, and is one dependent load per
        // level instead of a whole query in front of every sample launch (every lane walks the same point: broadcasts).
        float best = 3.402823466e+38f;
        {
            const float4* __restrict__ tv = (const float4*)mesh->triVerts;
            uint32_t w = 0u;
            for (int level = 0; level < 32; ++level)
            {
                const float4* q = wide + 8 * (size_t)w;
                const float4 hdr = __ldg(q), code = __ldg(q + 1), cu = __ldg(q + 2), cv = __ldg(q + 3), cn = __ldg(q + 4),
                             hu = __ldg(q + 5), hv = __ldg(q + 6), hn = __ldg(q + 7);
                const uint32_t ref[4] = { __float_as_uint(hdr.x), __float_as_uint(hdr.y), __float_as_uint(hdr.z), __float_as_uint(hdr.w) };
                uint32_t next = kNoNode;
                float nd = 3.402823466e+38f;
                #pragma unroll
                for (int k = 0; k < 4; ++k)
                {
                    const auto at = [k](const float4& v4) { return k == 0 ? v4.x : k == 1 ? v4.y : k == 2 ? v4.z : v4.w; };
                    F3 u, v, nrm;
                    decodeFrame(__float_as_uint(at(code)), u, v, nrm);
                    const float d = obbDist2(make_float4(at(cu), at(cv), at(cn), at(hu)), make_float4(u.x, u.y, u.z, at(hv)),
                                             make_float4(v.x, v.y, v.z, at(hn)), make_float4(nrm.x, nrm.y, nrm.z, 0.0f), c);
                    if (ref[k] != kNoNode && (next == kNoNode || d < nd)) { next = ref[k]; nd = d; }
                }
                if (next == kNoNode) break;
                if (next & 0x80000000u)
                {
                    const uint32_t first = next & 0x0FFFFFFFu, cnt = (next >> 28) & 7u;
                    for (uint32_t t = 0; t < cnt; ++t)
                    {
                        const float4 A = __ldg(tv + 3 * (size_t)(first + t)), B = __ldg(tv + 3 * (size_t)(first + t) + 1), C = __ldg(tv + 3 * (size_t)(first + t) + 2);
                        int sx, id;
                        const F3 cp = closestSimplex(c, f3(A.x, A.y, A.z), f3(B.x, B.y, B.z), f3(C.x, C.y, C.z), sx, id);
                        const F3 dv = sub3(c, cp);
                        best = fminf(best, dot3(dv, dv));
                    }
                    break;
                }
                w = next;
            }
        }
        const double dc = sqrt((double)best) * (1.0 + 1e-5) + eps;
        const double U = (dc + r) * (1.0 + 1e-5) + eps;

        // lanes 0-3: child `lane` of wide node w into `e`; returns whether it can hold a winner, with its lower bound
        uint32_t e[8];
        float lb = 0.0f;
        const auto child = [&](const uint32_t w) -> bool
        {
            if (lane >= 4u) return false;
            const float* rec = (const float*)(wide + 8 * (size_t)w);
            #pragma unroll
            for (int f = 0; f < 8; ++f) e[f] = __float_as_uint(__ldg(rec + 4 * f + lane));
            if (e[0] == kNoNode) return false;
            F3 u, v, nrm;
            decodeFrame(e[1], u, v, nrm);
            const auto gap = [&](const F3& a, int f)
            {
                const double q = cd[0] * a.x + cd[1] * a.y + cd[2] * a.z - (double)__uint_as_float(e[2 + f]);
                return fmax(fabs(q) - (double)__uint_as_float(e[5 + f]), 0.0);
            };
            const double gu = gap(u, 0), gv = gap(v, 1), gn = gap(nrm, 2);
            const double l = sqrt(gu * gu + gv * gv + gn * gn) * (1.0 - 2e-6) - r;
            lb = __double2float_rd(l);
            return l <= U;
        };
        // the root's children (all of them if none passes: then the bounds are not finite and the walk starts as from the root)
        bool keep = child(0u);
        unsigned mask = __ballot_sync(0xFFFFFFFFu, keep);
        if (!mask) { keep = lane < 4u && e[0] != kNoNode; mask = __ballot_sync(0xFFFFFFFFu, keep); lb = 0.0f; }
        if (keep)
        {
            const unsigned s = __popc(mask & ((1u << lane) - 1u));
            #pragma unroll
            for (int f = 0; f < 8; ++f) ent[s][f] = e[f];
            lbs[s] = lb; frozen[s] = 0;
        }
        unsigned count = __popc(mask), expanded = 0;
        __syncwarp();
        // best-first: replace the nearest inner entry by its children that can hold a winner, for as long as the cut stays
        // within kMeshCut entries; an entry whose children do not fit stays as it is
        for (int it = 0; it < 4 * kMeshCut; ++it)
        {
            float key = (lane < count && !(ent[lane][0] & 0x80000000u) && !frozen[lane]) ? lbs[lane] : 3.402823466e+38f;
            unsigned at = lane;
            #pragma unroll
            for (int s = 16; s > 0; s >>= 1)
            {
                const float k2 = __shfl_xor_sync(0xFFFFFFFFu, key, s);
                const unsigned a2 = __shfl_xor_sync(0xFFFFFFFFu, at, s);
                if (k2 < key || (k2 == key && a2 < at)) { key = k2; at = a2; }
            }
            if (!(key < 3.0e38f)) break;                                     // warp-uniform: no inner entry left to expand
            const uint32_t w = ent[at][0];
            keep = child(w);
            mask = __ballot_sync(0xFFFFFFFFu, keep);
            const unsigned ns = __popc(mask);
            __syncwarp();
            if (count - 1u + ns > (unsigned)kMeshCut)
            {
                if (lane == 0u) frozen[at] = 1;
                __syncwarp();
                continue;
            }
            // the first survivor takes the expanded entry's slot, the others are appended; none: the last entry moves there
            if (!ns && lane < 8u)
            {
                const uint32_t last = ent[count - 1u][lane];
                const float lastLb = lbs[count - 1u];
                const uint8_t lastFrozen = frozen[count - 1u];
                __syncwarp(0xFFu);
                ent[at][lane] = last;
                if (lane == 0u) { lbs[at] = lastLb; frozen[at] = lastFrozen; }
            }
            if (keep)
            {
                const unsigned rank = __popc(mask & ((1u << lane) - 1u));
                const unsigned s = rank ? count + rank - 1u : at;
                #pragma unroll
                for (int f = 0; f < 8; ++f) ent[s][f] = e[f];
                lbs[s] = lb; frozen[s] = 0;
            }
            count = count + ns - 1u;
            ++expanded;
            __syncwarp();
        }

        // nearest first (insertion sort of the entry order by lane 0), then one float of each record per lane
        if (lane == 0u)
        {
            uint8_t* ord = sOrd[wib];
            for (unsigned i = 0; i < count; ++i)
            {
                unsigned j = i;
                while (j > 0 && lbs[ord[j - 1]] > lbs[i]) { ord[j] = ord[j - 1]; --j; }
                ord[j] = (uint8_t)i;
            }
        }
        __syncwarp();
        const unsigned nrec = (count + 3u) / 4u;
        float* out = (float*)(cut + 8 * (size_t)fit * kCutStride);
        if (lane < 8u)
        {
            // record r > 0 gets the squared lower bound of its nearest entry (entries are sorted, so bounds grow with r) as
            // its stack bound: a sample whose bound is below it drops the record and every later one without reading them.
            // The bound carries the same relative 1e-5 and absolute eps as U, in the other direction.
            float rb[3];
            #pragma unroll
            for (int q = 0; q < 3; ++q)
            {
                const unsigned k = 4u * (q + 1u);
                const double l = k < count ? fmax((double)lbs[sOrd[wib][k]] * (1.0 - 1e-5) - eps, 0.0) : 0.0;
                rb[q] = __double2float_rd(l * l);
            }
            const float hdr[8] = { c.x, c.y, c.z, nextafterf((float)dc, 3.402823466e+38f), __uint_as_float(nrec), rb[0], rb[1], rb[2] };
            out[lane] = hdr[lane];
        }
        const unsigned f = lane >> 2;
        for (unsigned rr = 0; rr < nrec; ++rr)
        {
            const unsigned k = 4u * rr + (lane & 3u);
            uint32_t x;
            if (k < count) x = ent[sOrd[wib][k]][f];
            else x = f == 0u ? kNoNode : f == 1u ? kIdentityFrame : f < 5u ? 0u : __float_as_uint(-3.0e38f);     // putAbsentChild
            out[32 * (rr + 1u) + lane] = __uint_as_float(x);
        }
        if (stats && lane == 0u)
        {
            atomicAdd(stats + kCutStatWord, (unsigned long long)count);
            atomicMax(stats + kCutStatWord + 1, (unsigned long long)count);
            if (!expanded) atomicAdd(stats + kCutStatWord + 2, 1ull);
            atomicAdd(stats + kCutStatWord + 3, 1ull);
        }
    }

    __global__ void __launch_bounds__(256, 4)
    meshSampleKernel(const FitTask* __restrict__ tasks, unsigned long long nSamples, int D, const DeviceMeshView* __restrict__ mesh,
                     const RootMap map, const FitTablesDev tab, double* __restrict__ samples, unsigned long long* __restrict__ counter,
                     const unsigned grab, const int triThreshold,   // (triThreshold: see launchOne)
                     const int handOver,                            // 1 = tail phase on (0: diagnostics, HPSDF_MESH_NO_HANDOVER)
                     const float4* __restrict__ cutRec,             // meshCutKernel's records of these fits, or nullptr: start at the root, no seed (HPSDF_MESH_NO_CUT)
                     unsigned long long* __restrict__ stats)        // diagnostics (HPSDF_MESH_STATS): histogram of node steps per query and event
                                                                    // counts (kMeshStatCount x blockDim.x words of dynamic shared memory), or nullptr
    {
        // the leaf queues of the block, [slot][thread]: conflict-free, and out of the local memory that holds the stacks
        __shared__ unsigned long long sQueue[kMeshQueue][256];
        extern __shared__ unsigned sStat[];
        const float4* __restrict__ wide = (const float4*)mesh->wide;           // 8 float4 per 4-wide node (meshWideKernel)
        const float4* __restrict__ tv = (const float4*)mesh->triVerts;
        const double* __restrict__ roots = tab.roots[D];
        const unsigned n = (unsigned)fitRule(D), n2 = n * n, n3 = n2 * n;
        const unsigned lane = threadIdx.x & 31u, ltMask = (1u << lane) - 1u;

        // per-lane query state
        long long sid = -1;                       // sample index, -1 = idle
        F3 p = f3(0.0f, 0.0f, 0.0f);
        MeshHit h;
        float seed = 3.402823466e+38f;            // squared bound of the sample's distance from its fit's cut header (FLT_MAX: none)
        unsigned long long stack[kMeshStack];             // node | group << 28 | bound bits << 32
        int sp = 0;
        uint32_t cur = kNoNode; float curD = 0.0f;       // wide node (| group << 28) to process and its bound
        unsigned long long* const queue = &sQueue[0][threadIdx.x];  // circular, slot s at queue[s * 256]: head qh, count qn; entry = leaf reference | bound bits << 32
        int qh = 0, qn = 0;
        unsigned steps = 0;                                      // node steps of the lane's current query
        // warp-uniform work cursor
        unsigned long long cursor = 0, grabEnd = 0;
        bool exhausted = false;

        auto count = [&](const MeshStat c) { if (stats) ++sStat[c * blockDim.x + threadIdx.x]; };
        if (stats) for (int c = 0; c < kMeshStatCount; ++c) sStat[c * blockDim.x + threadIdx.x] = 0u;
        auto flushStats = [&]()
        {
            if (stats) for (int c = 0; c < kMeshStatCount; ++c) atomicAdd(stats + kMeshStatWord + c, (unsigned long long)sStat[c * blockDim.x + threadIdx.x]);
        };

        // One entry per call: a stale entry (its bound no longer beats the lane's best) is recognised by the next node step,
        // which drops it with its group and pops again — a divergent "skip the stale ones" loop here ran with 2-4 active lanes
        // and drew 29 % of the kernel's stall samples on its dependent local-memory loads.
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
            const bool wantNode = active && cur != kNoNode && qn <= kMeshQueue - 4;      // room for all four children being leaves
            const unsigned nodeMask = __ballot_sync(0xFFFFFFFFu, wantNode);
            const unsigned triMask = __ballot_sync(0xFFFFFFFFu, qn > 0);
            if (lane == 0 && (nodeMask == 0u || __popc(triMask) >= triThreshold) && triMask != 0u) count(kStatWarpTriIter);
            if (nodeMask != 0u && __popc(triMask) < triThreshold)
            {
                if (lane == 0) count(kStatWarpNodeIter);
                if (wantNode)
                {
                    ++steps;
                    const float lim = bound * 1.000001f;
                    if (curD > lim)
                    {
                        // went stale on the stack; so did the entries below it from the same node step (its farther siblings):
                        // drop them with it, no loads
                        const int group = (int)((cur >> kGroupShift) & 3u);
                        sp -= group;
                        count(kStatStalePop);
                        if (stats) sStat[kStatGroupDrop * blockDim.x + threadIdx.x] += (unsigned)group;
                        pop();
                    }
                    else
                    {
                        count(kStatNodeVisit);
                        // one cache line per step: the four child references, frame codes and boxes of the node, all requested at once
                        const float4* __restrict__ w = ((cur & kCutBit) ? cutRec : wide) + 8 * (size_t)(cur & kNodeIndexMask);
                        const float4 hdr = __ldg(w), code = __ldg(w + 1), cu = __ldg(w + 2), cv = __ldg(w + 3), cn = __ldg(w + 4),
                                     hu = __ldg(w + 5), hv = __ldg(w + 6), hn = __ldg(w + 7);
                        const uint32_t ref[4] = { __float_as_uint(hdr.x), __float_as_uint(hdr.y), __float_as_uint(hdr.z), __float_as_uint(hdr.w) };
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
                        // visit order: nearest first
                        uint32_t r[4] = { ref[0], ref[1], ref[2], ref[3] };
                        #define HPSDF_CSWAP(a, b) if (cd[b] < cd[a]) { const float td = cd[a]; cd[a] = cd[b]; cd[b] = td; const uint32_t tr = r[a]; r[a] = r[b]; r[b] = tr; }
                        HPSDF_CSWAP(0, 1) HPSDF_CSWAP(2, 3) HPSDF_CSWAP(0, 2) HPSDF_CSWAP(1, 3) HPSDF_CSWAP(1, 2)
                        #undef HPSDF_CSWAP
                        // leaves go straight to the queue, nearest first (wantNode left room for four)
                        #pragma unroll
                        for (int k = 0; k < 4; ++k)
                            if (cd[k] < 3.0e38f && (r[k] & 0x80000000u))
                            {
                                queue[((qh + qn) & (kMeshQueue - 1)) * 256] = stackEntry(r[k], cd[k]);   // 0x80000000 | count << 28 | first triangle slot
                                ++qn;
                            }
                        // inner children: the nearest becomes cur, the others go on the stack farthest first so that the nearest of
                        // them is popped next; each records how many of its farther siblings lie below it
                        uint32_t next = kNoNode, group = 0u;
                        float nextD = 0.0f;
                        #pragma unroll
                        for (int k = 3; k >= 0; --k)
                            if (cd[k] < 3.0e38f && !(r[k] & 0x80000000u))
                            {
                                if (next != kNoNode && sp < kMeshStack) { stack[sp++] = stackEntry(next | group << kGroupShift, nextD); ++group; }
                                next = r[k]; nextD = cd[k];
                            }
                        if (next != kNoNode) { cur = next | group << kGroupShift; curD = nextD; }
                        else pop();
                    }
                }
            }
            else if (qn > 0)
            {
                const unsigned long long e = queue[qh * 256];
                const uint32_t first = (uint32_t)e & 0x0FFFFFFFu, cnt = ((uint32_t)e >> 28) & 7u;
                if (__uint_as_float((uint32_t)(e >> 32)) <= bound * 1.000001f)    // else: pruned while it waited
                {
                    count(kStatLeafTest);
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
                else count(kStatLeafPruned);
                qh = (qh + 1) & (kMeshQueue - 1);
                --qn;
                // leaves the new best has pruned leave the queue now (shared-memory reads only), so that they neither take a
                // triangle iteration of their own nor count towards triThreshold. h.best is a distance this lane reached for
                // the same point, so it bounds the answer in the tail phase too.
                const float after = fminf(bound, h.best) * 1.000001f;
                while (qn > 0 && __uint_as_float((uint32_t)(queue[qh * 256] >> 32)) > after)
                {
                    count(kStatLeafPruned);
                    qh = (qh + 1) & (kMeshQueue - 1);
                    --qn;
                }
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
                    if (cutRec)
                    {
                        // start at the fit's first cut record, the others on the stack; seed the bound with
                        // d(x) <= dc + |x - c|, rounded up (meshCutKernel). Only a real triangle sets h.
                        const unsigned base = fit * (unsigned)kCutStride;
                        const float4 ch = __ldg(cutRec + 8 * (size_t)base);
                        const unsigned nrec = __float_as_uint(__ldg((const float*)(cutRec + 8 * (size_t)base + 1)));
                        const F3 dv = sub3(p, f3(ch.x, ch.y, ch.z));
                        const float bx = __fmul_rn(__fadd_rn(ch.w, __fsqrt_ru(dot3(dv, dv))), 1.00002f);
                        seed = fminf(__fmul_ru(bx, bx), 3.402823466e+38f);
                        // record rr with its bound (header words 5-7) and, as its group, the records after it: once it is
                        // stale, so are they
                        for (int rr = (int)nrec - 1; rr >= 1; --rr)
                            stack[sp++] = stackEntry((base + 1u + (unsigned)rr) | kCutBit | ((nrec - 1u - (unsigned)rr) << kGroupShift),
                                                     __ldg((const float*)(cutRec + 8 * (size_t)base + 1) + rr));
                        cur = (base + 1u) | kCutBit;
                    }
                }
                cursor += want < avail ? want : avail;
                idle = __ballot_sync(0xFFFFFFFFu, sid < 0);
            }
            if (idle == 0xFFFFFFFFu) { flushStats(); return; }                // nothing in flight and nothing left to take
            if (idle && handOver) break;                                      // no samples left and some lanes have nothing to do: tail phase
            step(true, fminf(h.best, seed));
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
        wBest[lane] = __float_as_uint(sid >= 0 ? seed : 3.402823466e+38f);     // the owner's seed (FLT_MAX: none)
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
            if (idle == 0xFFFFFFFFu) { flushStats(); return; }
            if (idle)
            {
                // the i-th lane without work takes the top stack entry of the i-th lane that has one to spare (only from lanes that
                // have seen a triangle: before that nothing can be pruned and a helper would walk its whole sub-tree); queued
                // leaves are not handed over
                const bool canGive = (sid >= 0 || owner >= 0) && sp > 0 && cur != kNoNode && h.best < 3.0e38f;
                const unsigned donors = __ballot_sync(0xFFFFFFFFu, canGive);
                if (donors)
                {
                    const int nPairs = min(__popc(idle), __popc(donors));
                    const bool take = sid < 0 && owner < 0 && (int)__popc(idle & ltMask) < nPairs;
                    const bool give = canGive && (int)__popc(donors & ltMask) < nPairs;
                    const int src = take ? (int)__fns(donors, 0u, __popc(idle & ltMask) + 1) : (int)lane;
                    uint32_t gN = kNoNode; float gD = 0.0f;
                    if (give)
                    {
                        --sp; const unsigned long long e = stack[sp]; gN = (uint32_t)e & (kNodeIndexMask | kCutBit); gD = __uint_as_float((uint32_t)(e >> 32)); ++helpers;
                        // the helper's stack starts empty (gN without group; a cut record stays one: record indices are global to
                        // the launch); if the entry was one of cur's siblings, cur's group lost it
                        if ((cur >> kGroupShift) & 3u) cur -= 1u << kGroupShift;
                    }
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
