// sched_kernels.cuh — the greedy build loop of Octree::Create on the device (state: sched.h, host driver: build_device.cpp).
//
// Reference: RunBuildThreadPool (Source/HP/Octree.cpp:194-309) + the decision of TickBuildThread (:558-659) with
// EstimateHImprovement / EstimatePImprovement (:804-856). One launch of schedRoundKernel per round (a single CTA of 1024
// threads: every step is a scan, a compaction or a histogram walk over a few thousand entries, and block-wide barriers cost
// 100x less than grid-wide ones):
//
//   ingest   the fit records of the round -> weighted errors of the 8 child fits and the p-fit of every evaluated job
//   passes   repeat: (a) from a sequential-greedy state, find the GUARANTEED LEVEL with the error histogram — taking the
//            queue in decreasing order e1 >= e2 >= ..., entry k is certain to be popped before termination if
//            total - (e1 + ... + e_{k-1}) >= threshold, because popping an entry and any of its descendants lowers the total
//            by at most that entry's error; descendants with a larger error are popped even earlier — and apply every
//            cached job at or above it in one data-parallel step (decision, child allocation by prefix sum, error
//            bookkeeping); (b) where the histogram guarantees nothing more, sort the head of the queue (up to 1024 entries)
//            and walk it exactly: with all head jobs cached and no new child overtaking the rest of the head, the prefix sums
//            of the exact decreases reproduce the sequential loop, including the step at which it terminates
//   select   warp-aggregated compaction of the open list; leaves at or above the level (plus the next-largest pending errors
//            up to min_round_jobs) become the jobs of the next round, grouped by degree with deterministic task positions
//
// Determinism: allocation offsets come from prefix sums in list order, histogram updates are integer atomics, floating-point
// reductions have a fixed shape — so the ranks of a multi-GPU build, which all run this kernel on replicated data, stay
// bit-identical without exchanging anything but fit results.
#pragma once
#include <cfloat>
#include "hp_common.h"
#include "sched.h"

namespace hpsdf
{
    // ---- keys and histogram buckets -----------------------------------------------------------------------------------
    __device__ __forceinline__ unsigned long long errKey(double e) { return e > 0.0 ? (unsigned long long)__double_as_longlong(e) : 0ull; }
    __device__ __forceinline__ int subOfKey(unsigned long long key) { return ((int)(key >> 52) + 78) * kSubPerOctave + (int)((key >> 48) & 15ull); }
    __device__ __forceinline__ double subLowerEdge(int sub)
    {
        const long long E = (long long)(sub / kSubPerOctave) - 78;
        if (E < 0) return 0.0;
        return __longlong_as_double((long long)(((unsigned long long)E << 52) | ((unsigned long long)(sub % kSubPerOctave) << 48)));
    }
    // integer upper bound of an error in units of 2^(max(E,1) - 1054): 32 significant bits, rounded up
    __device__ __forceinline__ unsigned long long errUnits(unsigned long long key)
    {
        const unsigned long long m = (key & 0xFFFFFFFFFFFFFull) | ((key >> 52) ? (1ull << 52) : 0ull);
        return (m >> 21) + 1ull;
    }
    __device__ __forceinline__ double subUnit(int sub)
    {
        const int E = sub / kSubPerOctave - 78;
        return ldexp(1.0, (E < 1 ? 1 : E) - 1054);
    }

    struct SchedShared
    {
        // working copies of the counters (written back at the end of the launch)
        uint32_t nNodes, nOpen, nJobs, nCached, poolUsed, done, topSub, nLog, nDecision, appliedP, appliedH, retired, nearTies;
        uint32_t passes, windowPasses, lastPassLogStart;
        double   total, exactSum, totalBeforeLast, lastTotal;
        unsigned long long levelKey;   // guaranteed level in force (error key; ~0 = sequential-greedy state, no level) ...
        uint32_t levelNode;            // ... and, for a level that splits a group of equal keys, the last node index included (kNone: all)
        int      aboveLevel;           // open entries at or above the level that are not refined yet
        // block-wide scratch
        double   warpD[32];
        uint32_t warpU[32];
        unsigned long long warpL[32];
        uint32_t tmpU[8];
        double   tmpD[4];
        int      tmpI[4];
        uint32_t degCnt[kMaxDegree + 2];     // fits per degree of the round being selected
        unsigned long long tPhase[4];        // globaltimer at the phase boundaries (diagnostics)
    };

    __device__ __forceinline__ unsigned long long globalTimerNs()
    {
        unsigned long long t;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
        return t;
    }

    // ---- block-wide primitives (1024 threads, fixed shape => deterministic floating-point results) -------------------------
    __device__ __forceinline__ uint32_t blockExclScanU(uint32_t v, uint32_t* sWarp, uint32_t& total)
    {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        uint32_t x = v;
        #pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o); if (lane >= o) x += y; }
        if (lane == 31) sWarp[warp] = x;
        __syncthreads();
        if (warp == 0)
        {
            uint32_t w = sWarp[lane];
            #pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, w, o); if (lane >= o) w += y; }
            sWarp[lane] = w;
        }
        __syncthreads();
        const uint32_t base = warp ? sWarp[warp - 1] : 0u;
        total = sWarp[31];
        __syncthreads();
        return base + x - v;
    }

    __device__ __forceinline__ double blockInclScanD(double v, double* sWarp, double& total)
    {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        double x = v;
        #pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const double y = __shfl_up_sync(0xFFFFFFFFu, x, o); if (lane >= o) x += y; }
        if (lane == 31) sWarp[warp] = x;
        __syncthreads();
        if (warp == 0)
        {
            double w = sWarp[lane];
            #pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const double y = __shfl_up_sync(0xFFFFFFFFu, w, o); if (lane >= o) w += y; }
            sWarp[lane] = w;
        }
        __syncthreads();
        const double base = warp ? sWarp[warp - 1] : 0.0;
        total = sWarp[31];
        __syncthreads();
        return base + x;
    }

    __device__ __forceinline__ uint32_t blockMinU(uint32_t v, uint32_t* sWarp)
    {
        #pragma unroll
        for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
        if ((threadIdx.x & 31) == 0) sWarp[threadIdx.x >> 5] = v;
        __syncthreads();
        uint32_t r = sWarp[threadIdx.x & 31];
        #pragma unroll
        for (int o = 16; o > 0; o >>= 1) r = min(r, __shfl_xor_sync(0xFFFFFFFFu, r, o));
        __syncthreads();
        return r;
    }

    __device__ __forceinline__ int blockSumI(int v, uint32_t* sWarp)
    {
        #pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
        if ((threadIdx.x & 31) == 0) sWarp[threadIdx.x >> 5] = (uint32_t)v;
        __syncthreads();
        int r = (int)sWarp[threadIdx.x & 31];
        #pragma unroll
        for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xFFFFFFFFu, r, o);
        __syncthreads();
        return r;
    }

    __device__ __forceinline__ unsigned long long blockSumL(unsigned long long v, unsigned long long* sWarp)
    {
        #pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
        if ((threadIdx.x & 31) == 0) sWarp[threadIdx.x >> 5] = v;
        __syncthreads();
        unsigned long long r = sWarp[threadIdx.x & 31];
        #pragma unroll
        for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xFFFFFFFFu, r, o);
        __syncthreads();
        return r;
    }

    constexpr unsigned long long kNoLevel = ~0ull;
    __device__ __forceinline__ bool atOrAbove(const SchedShared& sh, unsigned long long key, uint32_t node)
    {
        return sh.levelKey != kNoLevel && (key > sh.levelKey || (key == sh.levelKey && node <= sh.levelNode));
    }

    // Does a pending leaf join the next round? At or above the selection level: always. Top-up (min_round_jobs): sub-buckets above the
    // cut one whole, the cut sub-bucket by a hash of the node index with the share `cutTau` / 65536 — about as many leaves as the round
    // still wants, chosen independently per leaf (no ordering needed; a top-up job is speculation, any choice is valid).
    __device__ __forceinline__ bool selectsLeaf(double err, uint32_t node, double selLevel, int cutSub, uint32_t cutTau)
    {
        if (err >= selLevel) return true;
        const int sub = subOfKey(errKey(err));
        if (sub > cutSub) return true;
        return sub == cutSub && ((node * 2654435761u) >> 16) < cutTau;
    }

    // ---- histogram updates (integer atomics only) -------------------------------------------------------------------------
    __device__ __forceinline__ void histAdd(const SchedDev& S, SchedShared& sh, double e, bool pending)
    {
        const unsigned long long key = errKey(e);
        const int sub = subOfKey(key);
        atomicAdd(S.allCnt + sub, 1u);
        atomicAdd(S.allSum + sub, errUnits(key));
        if (pending) atomicAdd(S.pendCnt + sub, 1u);
        atomicMax(&sh.topSub, (uint32_t)sub);
    }
    __device__ __forceinline__ void histRemove(const SchedDev& S, double e)
    {
        const unsigned long long key = errKey(e);
        const int sub = subOfKey(key);
        atomicSub(S.allCnt + sub, 1u);
        atomicAdd(S.allSum + sub, 0ull - errUnits(key));
    }

    // ---- nearness weight (CalculatePolyWeighting / CalculateExpWeighting, Octree.cpp:1209-1247) ------------------------------------
    // The reference averages FApprox over 100 std::rand() points of the cell. Two deterministic statements of that estimate:
    //   HPSDF_NEARNESS_EXACT_MEAN: its limit, the exact cell mean c000 * NL[0][depth]^3;
    //   HPSDF_NEARNESS_MC_COUNTER: the estimator itself on Philox4x32-10 points (key = seed, counter = cell coordinates, depth, degree,
    //                              sample index) — the rule stated in include/hpsdf.h; the CPU checker runs the same rule through
    //                              the reference's own FApprox. FApprox (Octree.cpp:859-901) is mirrored operation by operation,
    //                              so the estimate differs from the checker's only through the 1e-15 relative difference of the
    //                              coefficients.
    // exp / pow are CUDA's: <= 2 ulp from the host libm, the same order as that difference.
    __device__ __noinline__ double nearnessMeanMc(const SchedDev& S, const double* __restrict__ c, uint32_t degree, float4 cell, uint32_t depth)
    {
        const float ctr[3] = { cell.x, cell.y, cell.z };
        const float ext = __fadd_rn(cell.w, cell.w);                                  // max - min of a dyadic cell: exact
        float mn[3];
        uint32_t ic[3];
        #pragma unroll
        for (int a = 0; a < 3; ++a)
        {
            mn[a] = __fsub_rn(ctr[a], cell.w);
            ic[a] = (uint32_t)__fmul_rn(__fadd_rn(mn[a], 0.5f), (float)(1u << depth));
        }
        const double scale = (double)(2u << depth);                                    // Octree.cpp:862
        const uint32_t nC = (uint32_t)coeffCount((int)degree);
        double sum = 0.0;
        for (uint32_t smp = 0; smp < 100u; ++smp)                                      // nSamples, Octree.cpp:1216, 1236
        {
            const Philox4 r = philox4x32_10(ic[0], ic[1], ic[2], depth | (degree << 8) | (smp << 16), (uint32_t)S.nearnessSeed, (uint32_t)(S.nearnessSeed >> 32));
            const uint32_t w[3] = { r.x, r.y, r.z };
            double lut[3][kMaxDegree + 1];
            #pragma unroll
            for (int a = 0; a < 3; ++a)
            {
                const float uf = __fmul_rn((float)(w[a] >> 8), 0x1p-24f);
                const float x = __fadd_rn(mn[a], __fmul_rn(ext, uf));                 // AlignedBox::sample(): min + (max - min) * u, f32
                const double u = __dmul_rn(__dsub_rn((double)x, (double)ctr[a]), scale);
                lut[a][0] = c_nl[0][depth];
                double m2 = 0.0, m1 = 1.0;
                for (uint32_t j = 1; j <= degree; ++j)
                {
                    const double l = __dsub_rn(__dmul_rn(__dmul_rn(c_rec[j][0], u), m1), __dmul_rn(c_rec[j][1], m2));      // Octree.cpp:879
                    m2 = m1; m1 = l;
                    lut[a][j] = __dmul_rn(l, c_nl[j][depth]);
                }
            }
            double f = 0.0;
            uint32_t idx = 0;
            for (uint32_t p = 0; p <= degree; ++p)                                     // BasisIndexValues order: shell p, then i, then j
                for (uint32_t i = 0; i <= p; ++i)
                    for (uint32_t j = 0; j <= p - i && idx < nC; ++j, ++idx)
                        f = __dadd_rn(f, __dmul_rn(c[idx], __dmul_rn(__dmul_rn(lut[0][i], lut[1][j]), lut[2][p - i - j])));      // Octree.cpp:891-897
            sum = __dadd_rn(sum, f);
        }
        return fabs(__ddiv_rn(sum, 100.0));
    }

    // coeffs / degree / cell: the fitted basis and its cell (only read in the mc_counter mode); c0 = coeffs[0] from the fit record
    __device__ __forceinline__ double nearnessWeightDev(const SchedDev& S, double c0, uint32_t depth, const double* __restrict__ coeffs, uint32_t degree, float4 cell)
    {
        if (S.nearnessType == HPSDF_NEARNESS_NONE) return 1.0;
        double m;
        if (S.nearnessMode == HPSDF_NEARNESS_MC_COUNTER) m = nearnessMeanMc(S, coeffs, degree, cell, depth);
        else
        {
            const double nl = c_nl[0][depth];
            m = fabs(__dmul_rn(c0, __dmul_rn(__dmul_rn(nl, nl), nl)));
        }
        const double d = sqrt(3.0);
        if (S.nearnessType == HPSDF_NEARNESS_POLYNOMIAL)
        {
            const double k = pow(__dsub_rn(1.0, __ddiv_rn(m, d)), S.nearnessStrength);
            const double kk = (k < 0.0) ? 0.0 : k;              // std::max<double>(k, 0.0)
            return (kk < 1.0) ? kk : 1.0;                        // std::min<double>(1.0, .)
        }
        return exp(__ddiv_rn(__dmul_rn(__dmul_rn(-1.0, S.nearnessStrength), m), d));
    }

    // the weighted error of fit c (0..7 children, 8 = the p-fit) of job j
    __device__ __forceinline__ double ingestFitError(const SchedDev& S, uint32_t j, uint32_t c, uint32_t node, uint32_t depth, uint8_t flags)
    {
        const float4 cell = S.cell[node];
        if (c < 8u)
        {
            const FitRecord r = S.recs[S.jobHPos[j] + c];
            const uint32_t deg = S.degree[node];
            const float q = cell.w * 0.5f;                                              // CornerAABB (Octree.cpp:1096-1112), as expandJobsDevKernel
            const float4 child = make_float4(cell.x + ((c & 1u) ? q : -q), cell.y + ((c & 2u) ? q : -q), cell.z + ((c & 4u) ? q : -q), q);
            return r.rawErr * nearnessWeightDev(S, r.c0, depth + 1, S.pool + S.jobHSlot[j] + (size_t)c * (size_t)coeffCount((int)deg), deg, child);
        }
        const FitRecord r = S.recs[S.jobPPos[j]];
        const uint32_t deg = (flags & 4u) ? (uint32_t)kCoarseDegree : (uint32_t)S.degree[node] + 1u;
        return r.rawErr * nearnessWeightDev(S, r.c0, depth, S.pool + S.jobPSlot[j], deg, cell);
    }

    // The h-vs-p decision of one cached job (Octree.cpp:600-601, 825, 854 with BASIS_MAX_DEGREE-1 -> maxDegree,
    // TREE_MAX_DEPTH -> maxDepth): kind 0 = the node leaves the queue, 1 = p-refinement, 2 = h-refinement.
    struct Decision
    {
        int    kind;
        double delta;       // decrease of the total: err - (sum of the new errors)
        double maxNew;      // largest new error
        double pImp, hImp;
        bool   nearTie;
        double margin;
    };

    __device__ __forceinline__ Decision decideJob(const SchedDev& S, uint32_t j, double err, uint32_t p, uint32_t depth)
    {
        Decision D;
        const double* E = S.jobErr + 9 * (size_t)j;
        const uint8_t flags = S.jobFlags[j];
        const bool doH = flags & 1u, doP = flags & 2u;
        double maxNew = 0.0, sumH = 0.0;
        #pragma unroll
        for (int i = 0; i < 8; ++i) { const double h = doH ? E[i] : 0.0; maxNew = (maxNew < h) ? h : maxNew; sumH = __dadd_rn(sumH, h); }
        const double pErr = doP ? E[8] : 0.0;
        D.hImp = doH ? __dmul_rn(__ddiv_rn(1.0, __dmul_rn(7.0, (double)coeffCount((int)p))), __dsub_rn(err, __dmul_rn(8.0, maxNew))) : 0.0;
        D.pImp = doP ? __dmul_rn(__ddiv_rn(1.0, (double)(coeffCount((int)p + 1) - coeffCount((int)p))), __dsub_rn(err, __dmul_rn(8.0, pErr))) : 0.0;
        const bool refineP = p < S.maxDegree && (depth == S.maxDepth || D.pImp > D.hImp);
        const bool refineH = depth < S.maxDepth && !refineP;
        D.kind = refineP ? 1 : (refineH ? 2 : 0);
        D.delta = refineP ? __dsub_rn(err, pErr) : (refineH ? __dsub_rn(err, sumH) : 0.0);
        D.maxNew = refineP ? pErr : (refineH ? maxNew : 0.0);
        D.nearTie = false; D.margin = 0.0;
        if (doH && doP)
        {
            const double mag = fmax(fabs(D.pImp), fabs(D.hImp));
            D.margin = mag > 0.0 ? fabs(D.pImp - D.hImp) / mag : 0.0;
            D.nearTie = D.margin <= 1e-9;
        }
        return D;
    }

    // Apply the cached jobs list[0 .. n) in list order (all threads call this). Body of the reference's output-drain loop
    // (Octree.cpp:245-297): degree / slot / error updates for P, Subdivide + 8 children for H, total bookkeeping, log.
    __device__ void applyJobs(const SchedDev& S, SchedShared& sh, const uint32_t* list, uint32_t n)
    {
        const int tid = threadIdx.x;
        for (uint32_t base = 0; base < n; base += kSchedThreads)
        {
            const uint32_t i = base + tid;
            const bool active = i < n;
            uint32_t j = kNone, node = 0, p = 0, depth = 0;
            double err = 0.0;
            Decision D;
            D.kind = 0; D.delta = 0.0; D.maxNew = 0.0; D.pImp = D.hImp = 0.0; D.nearTie = false; D.margin = 0.0;
            if (active)
            {
                j = list[i];
                node = S.jobNode[j]; p = S.degree[node]; depth = S.depth[node]; err = S.err[node];
                D = decideJob(S, j, err, p, depth);
            }
            uint32_t packedTotal = 0;
            const uint32_t packedOff = blockExclScanU((active && D.kind == 2 ? 8u : 0u) | (active && D.kind != 0 ? 1u << 16 : 0u), sh.warpU, packedTotal);
            const uint32_t childOff = packedOff & 0xFFFFu, logOff = packedOff >> 16;
            const uint32_t totalChildren = packedTotal & 0xFFFFu, totalLogged = packedTotal >> 16;
            double chunkDelta = 0.0;
            const double inclDelta = blockInclScanD(active ? D.delta : 0.0, sh.warpD, chunkDelta);
            const bool fits = sh.nNodes + totalChildren <= S.capNodes && sh.nOpen + totalChildren <= S.capNodes &&
                              sh.nLog + totalLogged <= S.capLog;
            if (!fits) { if (tid == 0) sh.done = 2u; __syncthreads(); return; }
            int aboveDelta = 0;
            if (active)
            {
                const double* E = S.jobErr + 9 * (size_t)j;
                S.jobFlags[j] |= 128u;
                S.jobOf[node] = kNone;
                histRemove(S, err);
                if (atOrAbove(sh, errKey(err), node)) --aboveDelta;
                if (D.kind == 1)
                {
                    const double pErr = E[8];
                    S.slot[node] = S.jobPSlot[j];                                              // Octree.cpp:286
                    S.degree[node] = (uint8_t)(p + 1);
                    S.err[node] = pErr;
                    S.state[node] = kStPending;                                                // back into the queue (Octree.cpp:289-290)
                    histAdd(S, sh, pErr, true);
                    if (atOrAbove(sh, errKey(pErr), node)) ++aboveDelta;
                }
                else if (D.kind == 2)
                {
                    const uint32_t c0 = sh.nNodes + childOff;                                  // Subdivide (Octree.cpp:1115-1128)
                    S.child[node] = c0;
                    S.degree[node] = kInternalTag;                                             // Octree.cpp:265-272
                    S.state[node] = kStInternal;
                    const float4 pc = S.cell[node];
                    const float q = pc.w * 0.5f;
                    const uint32_t hs = S.jobHSlot[j], nc = (uint32_t)coeffCount((int)p), code = S.code[node];
                    #pragma unroll
                    for (uint32_t c = 0; c < 8; ++c)
                    {
                        const uint32_t k = c0 + c;
                        S.cell[k] = make_float4(pc.x + ((c & 1u) ? q : -q), pc.y + ((c & 2u) ? q : -q), pc.z + ((c & 4u) ? q : -q), q);
                        S.child[k] = kNone;
                        S.slot[k] = hs + c * nc;                                               // Octree.cpp:275-290
                        S.err[k] = E[c];
                        S.code[k] = code | (c << (27 - 3 * (int)depth));
                        S.jobOf[k] = kNone;
                        S.depth[k] = (uint8_t)(depth + 1);
                        S.degree[k] = (uint8_t)p;
                        S.state[k] = kStPending;
                        S.open[sh.nOpen + childOff + c] = k;
                        histAdd(S, sh, E[c], true);
                        if (atOrAbove(sh, errKey(E[c]), k)) ++aboveDelta;
                    }
                }
                else S.state[node] = kStRetired;                                               // Octree.cpp:643-655
                if (D.kind != 0)
                {
                    hpsdf_apply_log_entry& L = S.log[sh.nLog + logOff];
                    L.node_idx = node; L.kind = D.kind == 1 ? 0u : 1u; L.degree = p; L.initial_err = err; L.new_err = D.maxNew;
                    L.p_improvement = D.pImp; L.h_improvement = D.hImp;
                    L.total_after = (S.totalMode == HPSDF_TOTAL_EXACT_SUM ? sh.exactSum : sh.total) - inclDelta;
                    if (logOff + 1 == totalLogged)                     // the last job of this chunk: the margins of the termination cut
                    {
                        sh.tmpD[0] = (S.totalMode == HPSDF_TOTAL_EXACT_SUM ? sh.exactSum : sh.total) - (inclDelta - D.delta);
                        sh.tmpD[1] = L.total_after;
                    }
                }
                if (D.nearTie)
                {
                    const uint32_t k = atomicAdd(&sh.nDecision, 1u);
                    if (k < S.capDecisions)
                    {
                        hpsdf_decision_log_entry& e = S.decisions[k];
                        const float4 pc = S.cell[node];
                        e.node_idx = node; e.depth = depth; e.degree = p; e.centre[0] = pc.x; e.centre[1] = pc.y; e.centre[2] = pc.z;
                        e.chose_p = D.kind == 1; e.kind = 0; e.p_improvement = D.pImp; e.h_improvement = D.hImp; e.relative_margin = D.margin;
                    }
                    atomicAdd(&sh.nearTies, 1u);
                }
            }
            // three counts in one reduction: P jobs | retired | (aboveDelta + 1) per thread
            const unsigned long long packedSum = blockSumL((unsigned long long)(active && D.kind == 1 ? 1u : 0u) | ((unsigned long long)(active && D.kind == 0 ? 1u : 0u) << 16) |
                                                           ((unsigned long long)(aboveDelta + 1) << 32), sh.warpL);
            const int nP = (int)(packedSum & 0xFFFFull), nR = (int)((packedSum >> 16) & 0xFFFFull), above = (int)(packedSum >> 32) - kSchedThreads;
            if (tid == 0)
            {
                sh.total -= chunkDelta; sh.exactSum -= chunkDelta;
                sh.nNodes += totalChildren; sh.nOpen += totalChildren; sh.nLog += totalLogged;
                sh.appliedP += (uint32_t)nP; sh.appliedH += totalChildren / 8u; sh.retired += (uint32_t)nR;
                sh.aboveLevel += above;
                if (totalLogged) { sh.totalBeforeLast = sh.tmpD[0]; sh.lastTotal = sh.tmpD[1]; }
            }
            __syncthreads();
        }
    }

    // Guaranteed level from the histogram (see the header comment). Returns the level (0 = everything, +inf = nothing);
    // countAbove = open entries at or above it.
    __device__ double histLevel(const SchedDev& S, SchedShared& sh, double value, uint32_t& countAbove)
    {
        const int tid = threadIdx.x;
        double remaining = value;
        uint32_t cntAbove = 0;
        for (int hi = (int)sh.topSub; hi >= 0; hi -= kSchedThreads)
        {
            const int idx = hi - tid;
            const uint32_t cnt = idx >= 0 ? S.allCnt[idx] : 0u;
            const double bound = cnt ? (double)S.allSum[idx] * subUnit(idx) * (1.0 + 1e-12) : 0.0;
            double chunkTotal = 0.0;
            const double incl = blockInclScanD(bound, sh.warpD, chunkTotal);
            const bool fail = cnt > 0u && !(remaining - incl >= S.threshold);
            const uint32_t firstFail = blockMinU(fail ? (uint32_t)tid : (uint32_t)kSchedThreads, sh.warpU);
            uint32_t total = 0;
            blockExclScanU((uint32_t)tid < firstFail ? cnt : 0u, sh.warpU, total);
            cntAbove += total;
            if (firstFail < (uint32_t)kSchedThreads)
            {
                countAbove = cntAbove;
                return subLowerEdge(hi - (int)firstFail + 1);            // upper edge of the sub-bucket the bound runs out in
            }
            remaining -= chunkTotal;
        }
        countAbove = cntAbove;
        return 0.0;
    }

    // ---- exact walk of the head of the queue ---------------------------------------------------------------------------
    struct WindowShared
    {
        unsigned long long key[kWindow];
        uint32_t           node[kWindow];
        uint32_t           hist[256];
        uint32_t           count;
    };

    // Smallest key such that at most kWindow open entries have key >= it, found with the sub-bucket histogram and, inside the
    // sub-bucket where the count crosses kWindow, by 8-bit refinement steps over the candidates of that sub-bucket. `limit`
    // (output) is kNone, or — when more than kWindow entries share the largest remaining key exactly — the number of those
    // to take in open-list order.
    __device__ unsigned long long windowCutoff(const SchedDev& S, SchedShared& sh, WindowShared& W, uint32_t& tieLimit)
    {
        const int tid = threadIdx.x;
        tieLimit = kNone;
        // 1. whole sub-buckets from the top
        uint32_t above = 0;
        int crossing = -1;
        for (int hi = (int)sh.topSub; hi >= 0 && crossing < 0; hi -= kSchedThreads)
        {
            const int idx = hi - tid;
            const uint32_t cnt = idx >= 0 ? S.allCnt[idx] : 0u;
            uint32_t total = 0;
            const uint32_t excl = blockExclScanU(cnt, sh.warpU, total);
            const bool over = cnt > 0u && above + excl + cnt > (uint32_t)kWindow;
            const uint32_t first = blockMinU(over ? (uint32_t)tid : (uint32_t)kSchedThreads, sh.warpU);
            if (first < (uint32_t)kSchedThreads)
            {
                if ((uint32_t)tid == first) { sh.tmpU[0] = above + excl; sh.tmpI[0] = idx; }
                __syncthreads();
                above = sh.tmpU[0]; crossing = sh.tmpI[0];
                __syncthreads();
            }
            else above += total;
        }
        if (crossing < 0) return 0ull;                                   // the whole queue fits into the window
        unsigned long long lowKey = errKey(subLowerEdge(crossing + 1));  // everything above the crossing sub-bucket is in
        if (above >= (uint32_t)kWindow / 4u) return lowKey;
        // 2. candidates of the crossing sub-bucket -> scratch
        if (tid == 0) W.count = 0;
        __syncthreads();
        for (uint32_t base = 0; base < sh.nOpen; base += kSchedThreads)
        {
            const uint32_t i = base + tid;
            bool in = false;
            uint32_t node = 0;
            if (i < sh.nOpen)
            {
                node = S.open[i];
                const uint8_t st = S.state[node];
                in = (st == kStPending || st == kStEval || st == kStCached) && subOfKey(errKey(S.err[node])) == crossing;
            }
            uint32_t total = 0;
            const uint32_t off = blockExclScanU(in ? 1u : 0u, sh.warpU, total);
            if (in) S.scratch[W.count + off] = node;                      // open-list order
            __syncthreads();
            if (tid == 0) W.count += total;
            __syncthreads();
        }
        const uint32_t nCand = W.count;
        // 3. refine 8 bits at a time: prefix = the bits of the crossing bin fixed so far
        unsigned long long prefix = errKey(subLowerEdge(crossing)) >> 48;    // exponent + 4 mantissa bits
        for (int shift = 40; shift >= 0; shift -= 8)
        {
            if (tid < 256) W.hist[tid] = 0;
            __syncthreads();
            for (uint32_t i = tid; i < nCand; i += kSchedThreads)
            {
                const unsigned long long k = errKey(S.err[S.scratch[i]]);
                if ((k >> (shift + 8)) == prefix) atomicAdd(&W.hist[(uint32_t)(k >> shift) & 255u], 1u);
            }
            __syncthreads();
            if (tid == 0)
            {
                int bin = 255;
                uint32_t cum = 0;
                while (bin >= 0 && above + cum + W.hist[bin] <= (uint32_t)kWindow) { cum += W.hist[bin]; --bin; }
                sh.tmpI[0] = bin;            // first bin that does not fit (-1: all fit)
                sh.tmpU[0] = cum;
            }
            __syncthreads();
            const int bin = sh.tmpI[0];
            const uint32_t cum = sh.tmpU[0];
            __syncthreads();
            if (bin < 0) return prefix << (shift + 8);
            above += cum;
            lowKey = ((prefix << 8) | (unsigned long long)(bin + 1)) << shift;       // keys above the crossing bin
            if (above >= (uint32_t)kWindow / 4u) return lowKey;
            prefix = (prefix << 8) | (unsigned long long)bin;
        }
        // more than kWindow - above entries share the key `prefix` exactly: take the first few in open-list order
        tieLimit = (uint32_t)kWindow - above;
        return prefix;
    }

    // One exact pass over the sorted head of the queue. Returns the number of jobs applied; sets sh.done on termination.
    __device__ uint32_t windowPass(const SchedDev& S, SchedShared& sh, WindowShared& W, double* sB /*[kWindow]*/, uint32_t* sList /*[kWindow]*/)
    {
        const int tid = threadIdx.x;
        const double value = S.totalMode == HPSDF_TOTAL_EXACT_SUM ? sh.exactSum : sh.total;
        uint32_t tieLimit = kNone;
        const unsigned long long lowKey = windowCutoff(S, sh, W, tieLimit);
        // gather the head: entries with key >= lowKey (ties at lowKey limited to tieLimit, in open-list order)
        if (tid == 0) { W.count = 0; sh.tmpU[1] = 0; }
        __syncthreads();
        for (uint32_t base = 0; base < sh.nOpen; base += kSchedThreads)
        {
            const uint32_t i = base + tid;
            bool in = false, tie = false;
            uint32_t node = 0;
            unsigned long long key = 0;
            if (i < sh.nOpen)
            {
                node = S.open[i];
                const uint8_t st = S.state[node];
                if (st == kStPending || st == kStEval || st == kStCached)
                {
                    key = errKey(S.err[node]);
                    in = key >= lowKey;
                    tie = tieLimit != kNone && key == lowKey;
                }
            }
            uint32_t tieTotal = 0;
            const uint32_t tieOff = blockExclScanU(tie ? 1u : 0u, sh.warpU, tieTotal);
            if (tie && sh.tmpU[1] + tieOff >= tieLimit) in = false;
            uint32_t total = 0;
            const uint32_t off = blockExclScanU(in ? 1u : 0u, sh.warpU, total);
            if (in && W.count + off < (uint32_t)kWindow)
            {
                W.key[W.count + off] = key; W.node[W.count + off] = node;
            }
            __syncthreads();
            if (tid == 0) { W.count = min(W.count + total, (uint32_t)kWindow); sh.tmpU[1] += tieTotal; }
            __syncthreads();
        }
        const uint32_t n = W.count;
        if (n == 0)
        {
            if (tid == 0) sh.done = 1u;                                      // nodeQueue.empty() (Octree.cpp:216)
            __syncthreads();
            return 0;
        }
        if ((uint32_t)tid >= n) { W.key[tid] = 0ull; W.node[tid] = kNone; }
        __syncthreads();
        // bitonic sort, descending by (key, then ascending node index): the reference's max-heap order; ties are its heap's accident
        for (uint32_t k = 2; k <= (uint32_t)kWindow; k <<= 1)
            for (uint32_t jj = k >> 1; jj > 0; jj >>= 1)
            {
                const uint32_t other = (uint32_t)tid ^ jj;
                if (other > (uint32_t)tid)
                {
                    const unsigned long long ka = W.key[tid], kb = W.key[other];
                    const uint32_t na = W.node[tid], nb = W.node[other];
                    const bool aFirst = ka > kb || (ka == kb && na < nb);          // a belongs before b in the final order
                    const bool up = ((uint32_t)tid & k) == 0;
                    if (up ? !aFirst : aFirst) { W.key[tid] = kb; W.key[other] = ka; W.node[tid] = nb; W.node[other] = na; }
                }
                __syncthreads();
            }
        // per entry: exact decrease if its job is cached and none of its new errors reaches the smallest key of the head
        const unsigned long long lastKey = W.key[n - 1];
        bool cachedHere = false, exactHere = false;
        double B = 0.0;
        uint32_t job = kNone;
        if ((uint32_t)tid < n)
        {
            const uint32_t node = W.node[tid];
            const double err = S.err[node];
            B = err;
            if (S.state[node] == kStCached)
            {
                job = S.jobOf[node];
                cachedHere = true;
                const Decision D = decideJob(S, job, err, S.degree[node], S.depth[node]);
                if (errKey(D.maxNew) < lastKey || D.kind == 0) { B = D.delta; exactHere = true; }
            }
        }
        double totalB = 0.0;
        const double inclB = blockInclScanD((uint32_t)tid < n ? B : 0.0, sh.warpD, totalB);
        const double before = value - (inclB - B);                                   // total before this entry is popped
        const bool ok = (uint32_t)tid < n && before >= S.threshold;
        const uint32_t firstStop = blockMinU(ok ? (uint32_t)kSchedThreads : (uint32_t)tid, sh.warpU);      // first entry that is not certain (n if all are)
        const uint32_t certain = min(firstStop, n);
        const uint32_t firstInexact = blockMinU(((uint32_t)tid < n && !exactHere) ? (uint32_t)tid : (uint32_t)kSchedThreads, sh.warpU);
        // termination: every entry before `certain` was handled exactly and the total is below the threshold there (Octree.cpp:216)
        const bool terminates = certain < n && firstInexact >= certain;
        // apply the certain cached entries in sorted order
        const bool take = (uint32_t)tid < certain && cachedHere;
        uint32_t nTake = 0;
        const uint32_t off = blockExclScanU(take ? 1u : 0u, sh.warpU, nTake);
        if (take) sList[off] = job;
        // the certain entries whose jobs are not cached yet keep the level in force until they are evaluated and applied
        const uint32_t waiting = certain - nTake;
        __syncthreads();
        if (tid == 0)
        {
            sh.windowPasses++;
            if (waiting) { sh.levelKey = W.key[certain - 1]; sh.levelNode = W.node[certain - 1]; sh.aboveLevel = (int)certain; }
        }
        __syncthreads();
        if (nTake)
        {
            if (tid == 0) sh.lastPassLogStart = sh.nLog;
            __syncthreads();
            applyJobs(S, sh, sList, nTake);
        }
        if (tid == 0)
        {
            if (!waiting) { sh.levelKey = kNoLevel; sh.levelNode = kNone; sh.aboveLevel = 0; }
            if (terminates && sh.done == 0u) sh.done = 1u;
        }
        __syncthreads();
        return nTake;
    }

    // ---- coarse stage (round 0) -----------------------------------------------------------------------------------------
    // All 16^3 cells sit in the reference's queue with err = 100 (Octree.cpp:176-177); each is popped, fitted at degree 2 and
    // pushed back with its real error (:228-238, :836-843). totalCoeffError starts at 8^4 * 100 (:212), so the first errors
    // added are rounded at ulp(4e5) = 5.8e-11 and the running total depends on the POP ORDER at the 1e-9 level (SURVEY.md F4).
    // That order is a property of std::priority_queue alone: every comparison the heap makes involves at least one key of
    // 100, or two re-pushed keys below 100 whose exchange moves no unfitted entry (build_device.cpp: coarsePopOrder derives it
    // once by running libstdc++'s push_heap / pop_heap on dummy keys) — so one thread replays the additions in that order.
    __device__ void coarseStage(const SchedDev& S, SchedShared& sh, const uint16_t* __restrict__ gOrder, double* sErr /*[4096]*/, double* sRun /*[4096]*/,
                                uint16_t* order /*[4096], shared*/)
    {
        const int tid = threadIdx.x;
        const uint32_t nJobs = 4096u;
        for (uint32_t k = tid; k < nJobs; k += kSchedThreads) order[k] = gOrder[k];
        bool bad = false;
        double localSum = 0.0;
        for (uint32_t j = tid; j < nJobs; j += kSchedThreads)
        {
            const uint32_t node = S.jobNode[j];
            const FitRecord r = S.recs[S.jobPPos[j]];
            const double e = r.rawErr * nearnessWeightDev(S, r.c0, S.depth[node], S.pool + S.jobPSlot[j], (uint32_t)kCoarseDegree, S.cell[node]);
            sErr[j] = e;
            bad |= !(e < kInitialErr);
            S.jobFlags[j] |= 128u;
            S.slot[node] = S.jobPSlot[j];
            S.degree[node] = (uint8_t)kCoarseDegree;
            S.err[node] = e;
            S.state[node] = kStPending;
            S.jobOf[node] = kNone;
            S.open[j] = node;
            histAdd(S, sh, e, true);
            localSum += e;
        }
        double tot = 0.0;
        blockInclScanD(localSum, sh.warpD, tot);
        const int anyBad = blockSumI(bad ? 1 : 0, sh.warpU);
        // the addends in pop order, computed by everybody; then one thread runs the dependent chain of 4096 additions
        for (uint32_t k = tid; k < nJobs; k += kSchedThreads) sRun[k] = sErr[order[k]] - kInitialErr;        // Octree.cpp:257: (pErr - err)
        __syncthreads();
        if (tid == 0)
        {
            double t = 4096.0 * kInitialErr;                                              // Octree.cpp:212
            for (uint32_t k0 = 0; k0 < nJobs; k0 += 8)
            {
                double x[8];
                #pragma unroll
                for (int u = 0; u < 8; ++u) x[u] = sRun[k0 + u];
                #pragma unroll
                for (int u = 0; u < 8; ++u) { t += x[u]; x[u] = t; }
                #pragma unroll
                for (int u = 0; u < 8; ++u) sRun[k0 + u] = x[u];
            }
            sh.total = t; sh.exactSum = tot; sh.lastTotal = t; sh.totalBeforeLast = nJobs > 1 ? sRun[nJobs - 2] : t;
            sh.nOpen = nJobs; sh.appliedP += nJobs; sh.nLog = nJobs;
            if (anyBad) sh.done = 3u;                                                     // an error >= 100 or NaN: the host scheduler takes over
        }
        __syncthreads();
        for (uint32_t k = tid; k < nJobs; k += kSchedThreads)
        {
            const uint32_t j = order[k];
            hpsdf_apply_log_entry& L = S.log[k];
            L.node_idx = S.jobNode[j]; L.kind = 0u; L.degree = 0u; L.initial_err = kInitialErr; L.new_err = sErr[j];
            L.p_improvement = sErr[j]; L.h_improvement = 0.0;                             // Octree.cpp:806-810, 836-843
            L.total_after = S.totalMode == HPSDF_TOTAL_EXACT_SUM ? INFINITY : sRun[k];
        }
        __syncthreads();
    }

    // ---- the round kernel ---------------------------------------------------------------------------------------------------
    constexpr size_t kSchedDynSmem = 2 * 4096 * sizeof(double) + 4096 * sizeof(uint16_t);   // coarse stage: errors + running totals + pop order; window: B + list

    __global__ void __launch_bounds__(kSchedThreads, 1) schedRoundKernel(const SchedDev S, const uint16_t* __restrict__ coarseOrder)
    {
        extern __shared__ double dyn[];
        __shared__ SchedShared sh;
        __shared__ WindowShared W;
        const int tid = threadIdx.x;
        SchedCounters& C = *S.ctr;
        if (tid == 0)
        {
            sh.nNodes = C.nNodes; sh.nOpen = C.nOpen; sh.nJobs = C.nJobs; sh.nCached = C.nCached; sh.poolUsed = C.poolUsed; sh.done = C.done;
            sh.topSub = C.topSub; sh.nLog = C.nLog; sh.nDecision = C.nDecision; sh.appliedP = C.appliedP; sh.appliedH = C.appliedH;
            sh.retired = C.retired; sh.nearTies = C.nearTies; sh.passes = C.passes; sh.windowPasses = C.windowPasses;
            sh.lastPassLogStart = C.lastPassLogStart;
            sh.total = C.total; sh.exactSum = C.exactSum; sh.totalBeforeLast = C.totalBeforeLast; sh.lastTotal = C.lastTotal;
            sh.levelKey = C.levelKey; sh.levelNode = C.levelNode; sh.aboveLevel = C.aboveLevel;
        }
        __syncthreads();
        const uint32_t round = C.round;
        if (tid == 0) sh.tPhase[0] = globalTimerNs();

        // ---- ingest ------------------------------------------------------------------------------------------------------
        if (round == 0) coarseStage(S, sh, coarseOrder, dyn, dyn + 4096, reinterpret_cast<uint16_t*>(dyn + 8192));
        else
        {
            const uint32_t j0 = C.roundJob0, nj = C.roundJobs;
            for (uint32_t item = tid; item < (S.split ? 0u : 9u * nj); item += kSchedThreads)          // one thread per (job, fit): 9 independent record reads per job (split mode: schedIngestKernel did it)
            {
                const uint32_t k = item / 9u, c = item - 9u * k;
                const uint32_t j = j0 + k, node = S.jobNode[j];
                const uint32_t depth = S.depth[node];
                const uint8_t flags = S.jobFlags[j];
                if (c < 8u)
                {
                    if (flags & 1u) S.jobErr[9 * (size_t)j + c] = ingestFitError(S, j, c, node, depth, flags);
                }
                else
                {
                    if (flags & 2u) S.jobErr[9 * (size_t)j + 8] = ingestFitError(S, j, 8u, node, depth, flags);
                    S.state[node] = kStCached;
                    S.cached[sh.nCached + k] = j;
                }
            }
            __syncthreads();
            if (tid == 0) sh.nCached += nj;
            __syncthreads();
        }

        // ---- passes ----------------------------------------------------------------------------------------------------
        if (tid == 0) sh.tPhase[3] = globalTimerNs();
        double* sB = dyn;
        uint32_t* sList = reinterpret_cast<uint32_t*>(dyn + kWindow);
        uint32_t* bulk = S.scratch + S.capNodes;                            // second half of the scratch: the jobs of a bulk pass
        for (uint32_t iter = 0; sh.done == 0u; ++iter)
        {
            if (tid == 0) { sh.passes++; if (iter > 1000000u) sh.done = 4u; }       // (a pass applies at least one job or ends the loop)
            __syncthreads();
            if (sh.done != 0u) break;
            if (sh.levelKey == kNoLevel)
            {
                // sequential-greedy state (Octree.cpp:216): terminated?
                const double value = S.totalMode == HPSDF_TOTAL_EXACT_SUM ? sh.exactSum : sh.total;
                // (every thread takes this decision from the same shared values; the barrier before the write keeps a thread that is
                // still reading sh.done above from seeing it — it would leave the loop through the other exit, one barrier out of step)
                if (!(value >= S.threshold) || sh.nOpen == 0u) { __syncthreads(); if (tid == 0) sh.done = 1u; __syncthreads(); break; }
                uint32_t cntAbove = 0;
                const double L = histLevel(S, sh, value, cntAbove);
                if (cntAbove > 0u)
                {
                    if (tid == 0) { sh.levelKey = errKey(L); sh.levelNode = kNone; sh.aboveLevel = (int)cntAbove; }
                    __syncthreads();
                }
                else
                {
                    // the histogram bound runs out inside the top sub-bucket: exact walk of the head
                    const uint32_t applied = windowPass(S, sh, W, sB, sList);
                    if (sh.done != 0u || applied == 0u) break;                  // terminated, or the head waits for evaluation
                    continue;
                }
            }
            // a level is in force: apply every cached job at or above it (any order gives the same tree)
            uint32_t nBulk = 0;
            for (uint32_t base = 0; base < sh.nCached; base += kSchedThreads * 4u)
            {
                uint32_t jv[4], mask = 0, cntHere = 0;
                #pragma unroll
                for (uint32_t r = 0; r < 4u; ++r)
                {
                    const uint32_t i = base + tid * 4u + r;
                    jv[r] = i < sh.nCached ? S.cached[i] : kNone;
                }
                #pragma unroll
                for (uint32_t r = 0; r < 4u; ++r)
                {
                    if (jv[r] == kNone || (S.jobFlags[jv[r]] & 128u)) continue;
                    const uint32_t node = S.jobNode[jv[r]];
                    if (atOrAbove(sh, errKey(S.err[node]), node)) { mask |= 1u << r; ++cntHere; }
                }
                uint32_t total = 0;
                uint32_t off = nBulk + blockExclScanU(cntHere, sh.warpU, total);
                #pragma unroll
                for (uint32_t r = 0; r < 4u; ++r) if (mask & (1u << r)) bulk[off++] = jv[r];
                nBulk += total;
            }
            __syncthreads();
            if (nBulk)
            {
                if (tid == 0) sh.lastPassLogStart = sh.nLog;
                __syncthreads();
                applyJobs(S, sh, bulk, nBulk);
            }
            if (sh.done != 0u) break;
            const int aboveNow = sh.aboveLevel;
            __syncthreads();                                                   // everybody has read it before thread 0 resets it
            if (aboveNow <= 0)
            {
                if (tid == 0) { sh.levelKey = kNoLevel; sh.levelNode = kNone; sh.aboveLevel = 0; }     // everything at or above the level is refined: sequential state again
                __syncthreads();
                continue;
            }
            if (nBulk == 0u) break;                                            // the rest of the level waits for evaluation
        }
        __syncthreads();

        // ---- select the next round + compact the lists ---------------------------------------------------------------------
        if (tid == 0) sh.tPhase[1] = globalTimerNs();
        uint32_t cnt[kMaxDegree + 2];
        #pragma unroll
        for (int d = 0; d <= kMaxDegree + 1; ++d) cnt[d] = 0;
        uint32_t nSel = 0;
        const uint32_t job0 = sh.nJobs;
        if (sh.done == 0u)
        {
            constexpr uint32_t IT = 8;                              // list entries per thread and chunk: one block-wide scan per 8192 entries
            // compact the cached list (drop applied jobs)
            uint32_t keep = 0;
            const uint32_t nCachedNow = sh.nCached;                 // (read once: thread 0 overwrites it right after the loop)
            for (uint32_t base = 0; base < nCachedNow; base += kSchedThreads * IT)
            {
                uint32_t jv[IT];
                uint32_t liveMask = 0, nl = 0;
                #pragma unroll
                for (uint32_t r = 0; r < IT; ++r)
                {
                    const uint32_t i = base + tid * IT + r;
                    jv[r] = i < nCachedNow ? S.cached[i] : kNone;
                }
                #pragma unroll
                for (uint32_t r = 0; r < IT; ++r)
                    if (jv[r] != kNone && !(S.jobFlags[jv[r]] & 128u)) { liveMask |= 1u << r; ++nl; }
                uint32_t total = 0;
                uint32_t off = keep + blockExclScanU(nl, sh.warpU, total);
                #pragma unroll
                for (uint32_t r = 0; r < IT; ++r) if (liveMask & (1u << r)) S.cached[off++] = jv[r];
                keep += total;
                __syncthreads();
            }
            __syncthreads();
            if (tid == 0) sh.nCached = keep;
            if (tid < kMaxDegree + 2) sh.degCnt[tid] = 0;
            __syncthreads();

            // (a level that splits a group of equal keys selects the whole group: evaluating a leaf early changes nothing)
            double selLevel = sh.levelKey != kNoLevel ? __longlong_as_double((long long)sh.levelKey) : 0.0;
            for (uint32_t k = 0; k < S.speculate; ++k) selLevel *= 0.125;
            // top-up: the sub-bucket in which the count of pending leaves reaches minRoundJobs; it is taken whole (its errors
            // lie within 6 % of each other: the greedy loop is about to reach all of them)
            int cutSub = 0x7FFFFFFF;
            uint32_t cutTau = 65536u;                               // share of the cut sub-bucket that is taken, in 1/65536 (by a hash of the node index)
            if (S.minRoundJobs > 1u)
            {
                uint32_t above = 0;
                bool found = false;
                for (int hi = (int)sh.topSub; hi >= 0 && !found; hi -= kSchedThreads)
                {
                    const int idx = hi - tid;
                    const uint32_t pc = idx >= 0 ? S.pendCnt[idx] : 0u;
                    uint32_t total = 0;
                    const uint32_t excl = blockExclScanU(pc, sh.warpU, total);
                    const bool reach = pc > 0u && above + excl + pc >= S.minRoundJobs;
                    const uint32_t first = blockMinU(reach ? (uint32_t)tid : (uint32_t)kSchedThreads, sh.warpU);
                    if (first < (uint32_t)kSchedThreads)
                    {
                        if ((uint32_t)tid == first)
                        {
                            const uint32_t need = S.minRoundJobs - (above + excl);           // leaves wanted from this sub-bucket, of pc
                            sh.tmpU[0] = (uint32_t)min(65536ull, ((unsigned long long)need * 65536ull + pc - 1u) / pc);
                        }
                        __syncthreads();
                        cutSub = hi - (int)first; cutTau = sh.tmpU[0]; found = true;
                        __syncthreads();
                    }
                    else above += total;
                }
                if (!found) cutSub = 0;                             // fewer pending leaves than minRoundJobs: all of them
            }
            uint32_t lay2Begin[kMaxDegree + 2], lay2Pool[kMaxDegree + 2];
            for (int d = 0; d <= kMaxDegree + 1; ++d) { lay2Begin[d] = 0; lay2Pool[d] = sh.poolUsed; }
            if (S.split)
            {
                // the multi-block selection kernels take it from here (schedSelectCountKernel / schedSelectScatterKernel)
                if (tid == 0) { C.selLevel = selLevel; C.selCutSub = cutSub; C.selCutTau = cutTau; C.selOpen = sh.nOpen; C.selJob0 = job0; C.selPool0 = sh.poolUsed; }
                __syncthreads();
            }
            else
            {
                // pass A over the open list: compaction (dead entries out) + selection. Offsets come from one block-wide scan of
                // packed per-thread counts (warp shuffles + one exchange through shared memory), so list order is preserved.
                uint32_t keepOpen = 0;
                const uint32_t nOpenNow = sh.nOpen;                 // (read once: thread 0 overwrites it right after the loop)
                for (uint32_t base = 0; base < nOpenNow; base += kSchedThreads * IT)
                {
                    uint32_t nv[IT];
                    double ev[IT];
                    uint32_t liveMask = 0, selMask = 0, nl = 0, ns = 0;
                    #pragma unroll
                    for (uint32_t r = 0; r < IT; ++r)
                    {
                        const uint32_t i = base + tid * IT + r;
                        nv[r] = i < nOpenNow ? S.open[i] : kNone;
                    }
                    #pragma unroll
                    for (uint32_t r = 0; r < IT; ++r)
                    {
                        ev[r] = 0.0;
                        if (nv[r] == kNone) continue;
                        const uint8_t st = S.state[nv[r]];
                        if (st == kStPending || st == kStEval || st == kStCached) { liveMask |= 1u << r; ++nl; }
                        if (st == kStPending)
                        {
                            ev[r] = S.err[nv[r]];
                            if (selectsLeaf(ev[r], nv[r], selLevel, cutSub, cutTau)) { selMask |= 1u << r; ++ns; }
                        }
                    }
                    uint32_t total = 0;
                    const uint32_t excl = blockExclScanU(nl | (ns << 16), sh.warpU, total);
                    uint32_t lo = keepOpen + (excl & 0xFFFFu), so = nSel + (excl >> 16);
                    #pragma unroll
                    for (uint32_t r = 0; r < IT; ++r)
                    {
                        if (liveMask & (1u << r)) S.open[lo++] = nv[r];
                        if (selMask & (1u << r))
                        {
                            const uint32_t j = job0 + so++;
                            if (j < S.capJobs)
                            {
                                const uint32_t node = nv[r], p = S.degree[node], depth = S.depth[node];
                                const uint8_t flags = (uint8_t)((depth < S.maxDepth ? 1u : 0u) | (p < S.maxDegree ? 2u : 0u));    // Octree.cpp:600-601: fits that can never be used are skipped
                                S.jobNode[j] = node; S.jobFlags[j] = flags;
                                S.jobOf[node] = j;
                                S.state[node] = kStEval;
                                atomicSub(S.pendCnt + subOfKey(errKey(ev[r])), 1u);
                                if (flags & 1u) atomicAdd(&sh.degCnt[p], 8u);
                                if (flags & 2u) atomicAdd(&sh.degCnt[p + 1], 1u);
                            }
                        }
                    }
                    keepOpen += total & 0xFFFFu; nSel += total >> 16;
                    __syncthreads();
                }
                if (tid == 0) sh.nOpen = keepOpen;
                if (job0 + nSel > S.capJobs) { if (tid == 0) sh.done = 2u; nSel = 0; }
                __syncthreads();
                for (int d = 1; d <= kMaxDegree; ++d) cnt[d] = nSel ? sh.degCnt[d] : 0u;
                uint32_t groupBegin[kMaxDegree + 2], groupPool[kMaxDegree + 2];
                uint64_t poolNeed = 0;
                layoutRound(cnt, sh.poolUsed, groupBegin, groupPool, poolNeed);
                if (poolNeed >= 0xFFFFFFF0ull) { if (tid == 0) sh.done = 2u; nSel = 0; }
                for (int d = 0; d <= kMaxDegree + 1; ++d) { lay2Begin[d] = groupBegin[d]; lay2Pool[d] = groupPool[d]; }
                __syncthreads();
                // positions of every job's fits inside its groups, in job order; job records for expandJobsDevKernel
                uint32_t cursor[kMaxDegree + 2];
                for (int d = 0; d <= kMaxDegree + 1; ++d) cursor[d] = groupBegin[d];
                // several GPUs: task positions are handed out along the deal permutation of the round's jobs (dealStride; only pool
                // slots and record positions depend on it)
                uint32_t stride = 1u;
                if (S.dealJobs && nSel > 2u) stride = dealStride(nSel);
                for (uint32_t base = 0; base < nSel; base += kSchedThreads * 4u)
                {
                    uint32_t node[4], p[4], hPos[4], pPos[4];
                    uint8_t flags[4];
                    #pragma unroll
                    for (uint32_t r = 0; r < 4u; ++r)
                    {
                        const uint32_t k = base + tid * 4u + r;
                        node[r] = 0; p[r] = 0; flags[r] = 0; hPos[r] = 0; pPos[r] = 0;
                        if (k < nSel) { const uint32_t j = job0 + (uint32_t)(((unsigned long long)k * stride) % nSel); node[r] = S.jobNode[j]; p[r] = S.degree[node[r]]; flags[r] = S.jobFlags[j]; }
                    }
                    for (int d = 1; d <= kMaxDegree; ++d)
                    {
                        if (!cnt[d]) continue;
                        uint32_t mine = 0;
                        #pragma unroll
                        for (uint32_t r = 0; r < 4u; ++r)
                            mine += ((flags[r] & 1u) && p[r] == (uint32_t)d) ? 8u : (((flags[r] & 2u) && p[r] + 1u == (uint32_t)d) ? 1u : 0u);
                        uint32_t total = 0;
                        uint32_t off = cursor[d] + blockExclScanU(mine, sh.warpU, total);
                        #pragma unroll
                        for (uint32_t r = 0; r < 4u; ++r)
                        {
                            if ((flags[r] & 1u) && p[r] == (uint32_t)d) { hPos[r] = off; off += 8u; }
                            else if ((flags[r] & 2u) && p[r] + 1u == (uint32_t)d) { pPos[r] = off; off += 1u; }
                        }
                        cursor[d] += total;
                    }
                    #pragma unroll
                    for (uint32_t r = 0; r < 4u; ++r)
                    {
                        const uint32_t k = base + tid * 4u + r;
                        if (k >= nSel) continue;
                        const uint32_t j = job0 + (uint32_t)(((unsigned long long)k * stride) % nSel), pp = p[r];
                        const uint32_t depth = S.depth[node[r]];
                        S.jobHPos[j] = hPos[r]; S.jobPPos[j] = pPos[r];
                        S.jobHSlot[j] = (flags[r] & 1u) ? groupPool[pp] + (hPos[r] - groupBegin[pp]) * (uint32_t)coeffCount((int)pp) : 0u;
                        S.jobPSlot[j] = (flags[r] & 2u) ? groupPool[pp + 1] + (pPos[r] - groupBegin[pp + 1]) * (uint32_t)coeffCount((int)pp + 1) : 0u;
                        const float4 c = S.cell[node[r]];
                        JobDesc o;
                        o.cx = c.x; o.cy = c.y; o.cz = c.z; o.half = c.w;
                        o.hPos = hPos[r]; o.pPos = pPos[r]; o.src = S.slot[node[r]];
                        o.depth = (uint8_t)depth; o.degree = (uint8_t)pp; o.flags = flags[r]; o.pad = 0;
                        S.jobsOut[k] = o;
                    }
                }
            }
            if (tid == 0 && !S.split)
            {
                RoundLayout lay;
                for (int d = 0; d <= kMaxDegree + 1; ++d) { lay.groupBegin[d] = lay2Begin[d]; lay.groupPool[d] = lay2Pool[d]; }
                *S.layout = lay;
                if (sh.done == 0u) { sh.poolUsed = lay2Pool[kMaxDegree + 1]; sh.nJobs = job0 + nSel; }
                if (nSel == 0u && sh.done == 0u) sh.done = 4u;               // nothing to evaluate and not terminated: internal error
            }
            __syncthreads();
        }

        // ---- write back + header -------------------------------------------------------------------------------------------
        if (tid == 0)
        {
            uint32_t nTasks = 0;
            for (int d = 1; d <= kMaxDegree; ++d) nTasks += cnt[d];
            C.nNodes = sh.nNodes; C.nOpen = sh.nOpen; C.nJobs = sh.nJobs; C.nCached = sh.nCached; C.poolUsed = sh.poolUsed; C.done = sh.done;
            C.topSub = sh.topSub; C.nLog = sh.nLog; C.nDecision = sh.nDecision; C.appliedP = sh.appliedP; C.appliedH = sh.appliedH;
            C.retired = sh.retired; C.nearTies = sh.nearTies; C.passes = sh.passes; C.windowPasses = sh.windowPasses;
            C.lastPassLogStart = sh.lastPassLogStart;
            C.total = sh.total; C.exactSum = sh.exactSum; C.totalBeforeLast = sh.totalBeforeLast; C.lastTotal = sh.lastTotal;
            C.roundJob0 = job0; C.roundJobs = sh.done == 0u ? nSel : 0u;
            C.jobsEvaluated += sh.done == 0u ? nSel : 0u; C.fitsEvaluated += sh.done == 0u ? nTasks : 0u;
            C.round = round + 1;
            const unsigned long long tEnd = globalTimerNs();
            C.nsIngest += sh.tPhase[3] - sh.tPhase[0]; C.nsPasses += sh.tPhase[1] - sh.tPhase[3]; C.nsSelect += tEnd - sh.tPhase[1];
            C.levelKey = sh.levelKey; C.levelNode = sh.levelNode; C.aboveLevel = sh.aboveLevel;
            if (!(S.split && sh.done == 0u))               // split mode: the selection kernel publishes the header of a round that goes on
            {
                RoundHeader* H = S.hostHdr;
                H->done = sh.done; H->nJobs = sh.done == 0u ? nSel : 0u; H->nTasks = sh.done == 0u ? nTasks : 0u;
                for (int d = 0; d <= kMaxDegree + 1; ++d) H->cnt[d] = sh.done == 0u ? cnt[d] : 0u;
                H->nNodes = sh.nNodes; H->nOpen = sh.nOpen; H->nCached = sh.nCached; H->poolUsed = sh.poolUsed;
                __threadfence_system();
                H->seq = round + 1;
                __threadfence_system();
            }
        }
    }

    // ---- split mode: ingest and selection as multi-block kernels around the single-CTA pass kernel -------------------------------
    // (single GPU; several GPUs deal the jobs out along a stride permutation, which the single-CTA selection above does)
    __global__ void __launch_bounds__(256) schedIngestKernel(const SchedDev S)
    {
        const SchedCounters& C = *S.ctr;
        const uint32_t j0 = C.roundJob0, nj = C.roundJobs, nCached = C.nCached;
        const uint32_t item = blockIdx.x * blockDim.x + threadIdx.x;
        if (item >= 9u * nj) return;
        const uint32_t k = item / 9u, c = item - 9u * k;
        const uint32_t j = j0 + k, node = S.jobNode[j];
        const uint32_t depth = S.depth[node];
        const uint8_t flags = S.jobFlags[j];
        if (c < 8u)
        {
            if (flags & 1u) S.jobErr[9 * (size_t)j + c] = ingestFitError(S, j, c, node, depth, flags);
        }
        else
        {
            if (flags & 2u) S.jobErr[9 * (size_t)j + 8] = ingestFitError(S, j, 8u, node, depth, flags);
            S.state[node] = kStCached;
            S.cached[nCached + k] = j;
        }
    }


    // what one thread sees of its kSelItems consecutive open-list entries
    struct SelView
    {
        uint32_t node[kSelItems];
        double   err[kSelItems];
        uint32_t liveMask, selMask, nLive, nSel;
    };
    __device__ __forceinline__ void selLoad(const SchedDev& S, const SchedCounters& C, uint32_t chunk, SelView& V)
    {
        const uint32_t base = chunk * kSelChunk + threadIdx.x * kSelItems;
        V.liveMask = V.selMask = V.nLive = V.nSel = 0;
        #pragma unroll
        for (uint32_t r = 0; r < kSelItems; ++r) V.node[r] = base + r < C.selOpen ? S.open[base + r] : kNone;
        #pragma unroll
        for (uint32_t r = 0; r < kSelItems; ++r)
        {
            V.err[r] = 0.0;
            if (V.node[r] == kNone) continue;
            const uint8_t st = S.state[V.node[r]];
            if (st == kStPending || st == kStEval || st == kStCached) { V.liveMask |= 1u << r; ++V.nLive; }
            if (st == kStPending)
            {
                V.err[r] = S.err[V.node[r]];
                if (selectsLeaf(V.err[r], V.node[r], C.selLevel, C.selCutSub, C.selCutTau)) { V.selMask |= 1u << r; ++V.nSel; }
            }
        }
    }

    // pass 1: per chunk of kSelChunk entries: live entries, selected entries, fits per degree -> chunkCounts[chunk][16]
    __global__ void __launch_bounds__(kSchedThreads, 1) schedSelectCountKernel(const SchedDev S)
    {
        __shared__ uint32_t sCnt[16];
        const SchedCounters& C = *S.ctr;
        if (C.done != 0u) return;
        const uint32_t nChunks = (C.selOpen + kSelChunk - 1) / kSelChunk;
        for (uint32_t chunk = blockIdx.x; chunk < nChunks; chunk += gridDim.x)
        {
            if (threadIdx.x < 16) sCnt[threadIdx.x] = 0;
            __syncthreads();
            SelView V;
            selLoad(S, C, chunk, V);
            #pragma unroll
            for (uint32_t r = 0; r < kSelItems; ++r)
                if (V.selMask & (1u << r))
                {
                    const uint32_t node = V.node[r], p = S.degree[node], depth = S.depth[node];
                    if (depth < S.maxDepth) atomicAdd(&sCnt[2 + p], 8u);
                    if (p < S.maxDegree) atomicAdd(&sCnt[2 + p + 1], 1u);
                }
            uint32_t packed = V.nLive | (V.nSel << 16);
            #pragma unroll
            for (int o = 16; o > 0; o >>= 1) packed += __shfl_xor_sync(0xFFFFFFFFu, packed, o);
            if ((threadIdx.x & 31) == 0) { atomicAdd(&sCnt[0], packed & 0xFFFFu); atomicAdd(&sCnt[1], packed >> 16); }
            __syncthreads();
            if (threadIdx.x < 16) S.chunkCounts[chunk * 16 + threadIdx.x] = sCnt[threadIdx.x];
            __syncthreads();
        }
    }

    // pass 2: offsets from the chunk counts; compacted open list -> openAlt; the selected leaves become jobs with deterministic task
    // positions (list order); block 0 publishes the round: layout, counters, header
    __global__ void __launch_bounds__(kSchedThreads, 1) schedSelectScatterKernel(const SchedDev S)
    {
        __shared__ uint32_t sBase[16], sTotal[16], sWarp[32];
        SchedCounters& C = *S.ctr;
        if (C.done != 0u) return;
        const uint32_t tid = threadIdx.x;
        const uint32_t nChunks = (C.selOpen + kSelChunk - 1) / kSelChunk;
        const uint32_t job0 = C.selJob0, poolUsed0 = C.selPool0, round = C.round;           // (the pass kernel already advanced `round`)
        for (uint32_t chunk = blockIdx.x; chunk < (nChunks ? nChunks : 1u); chunk += gridDim.x)
        {
            // totals over all chunks and the sums over the chunks before this one, 16 counters each
            if (tid < 16) { sBase[tid] = 0; sTotal[tid] = 0; }
            __syncthreads();
            for (uint32_t e = tid; e < nChunks * 16u; e += kSchedThreads)
            {
                const uint32_t v = S.chunkCounts[e];
                if (v) { atomicAdd(&sTotal[e & 15u], v); if ((e >> 4) < chunk) atomicAdd(&sBase[e & 15u], v); }
            }
            __syncthreads();
            const uint32_t nSel = sTotal[1];
            uint32_t groupBegin[kMaxDegree + 2], groupPool[kMaxDegree + 2];
            uint64_t poolNeed = 0;
            const uint32_t nTasks = layoutRound(sTotal + 2, poolUsed0, groupBegin, groupPool, poolNeed);
            const bool overflow = job0 + nSel > S.capJobs || poolNeed >= 0xFFFFFFF0ull;
            const uint32_t doneCode = overflow ? 2u : (nSel == 0u ? 4u : 0u);
            if (chunk == 0 && tid == 0)
            {
                // publish the round (the pass kernel left the header alone)
                RoundLayout lay;
                for (int d = 0; d <= kMaxDegree + 1; ++d) { lay.groupBegin[d] = groupBegin[d]; lay.groupPool[d] = groupPool[d]; }
                *S.layout = lay;
                RoundHeader* H = S.hostHdr;
                H->done = doneCode; H->nJobs = doneCode ? 0u : nSel; H->nTasks = doneCode ? 0u : nTasks;
                for (int d = 0; d <= kMaxDegree + 1; ++d) H->cnt[d] = (doneCode || d < 1 || d > kMaxDegree) ? 0u : sTotal[2 + d];
                H->nNodes = C.nNodes; H->nOpen = sTotal[0]; H->nCached = C.nCached; H->poolUsed = doneCode ? poolUsed0 : (uint32_t)poolNeed;
                __threadfence_system();
                H->seq = round;
                __threadfence_system();
            }
            if (doneCode) { if (chunk == 0 && tid == 0) C.done = doneCode; return; }
            SelView V;
            selLoad(S, C, chunk, V);
            // offsets inside the chunk (list order)
            uint32_t total = 0;
            const uint32_t excl = blockExclScanU(V.nLive | (V.nSel << 16), sWarp, total);
            uint32_t lo = sBase[0] + (excl & 0xFFFFu), so = sBase[1] + (excl >> 16);
            uint32_t p[kSelItems], hPos[kSelItems], pPos[kSelItems];
            uint8_t flags[kSelItems];
            #pragma unroll
            for (uint32_t r = 0; r < kSelItems; ++r)
            {
                p[r] = 0; flags[r] = 0; hPos[r] = 0; pPos[r] = 0;
                if (V.selMask & (1u << r))
                {
                    const uint32_t node = V.node[r];
                    p[r] = S.degree[node];
                    flags[r] = (uint8_t)((S.depth[node] < S.maxDepth ? 1u : 0u) | (p[r] < S.maxDegree ? 2u : 0u));    // Octree.cpp:600-601
                }
            }
            for (int d = 1; d <= kMaxDegree; ++d)
            {
                if (!S.chunkCounts[chunk * 16 + 2 + d]) continue;                       // no fit of this degree in this chunk
                uint32_t mine = 0;
                #pragma unroll
                for (uint32_t r = 0; r < kSelItems; ++r)
                    mine += ((flags[r] & 1u) && p[r] == (uint32_t)d) ? 8u : (((flags[r] & 2u) && p[r] + 1u == (uint32_t)d) ? 1u : 0u);
                uint32_t t2 = 0;
                uint32_t off = groupBegin[d] + sBase[2 + d] + blockExclScanU(mine, sWarp, t2);
                #pragma unroll
                for (uint32_t r = 0; r < kSelItems; ++r)
                {
                    if ((flags[r] & 1u) && p[r] == (uint32_t)d) { hPos[r] = off; off += 8u; }
                    else if ((flags[r] & 2u) && p[r] + 1u == (uint32_t)d) { pPos[r] = off; off += 1u; }
                }
            }
            #pragma unroll
            for (uint32_t r = 0; r < kSelItems; ++r)
            {
                if (V.liveMask & (1u << r)) S.openAlt[lo++] = V.node[r];
                if (!(V.selMask & (1u << r))) continue;
                const uint32_t k = so++, j = job0 + k, node = V.node[r], pp = p[r];
                S.jobNode[j] = node; S.jobFlags[j] = flags[r];
                S.jobOf[node] = j;
                S.state[node] = kStEval;
                atomicSub(S.pendCnt + subOfKey(errKey(V.err[r])), 1u);
                S.jobHPos[j] = hPos[r]; S.jobPPos[j] = pPos[r];
                S.jobHSlot[j] = (flags[r] & 1u) ? groupPool[pp] + (hPos[r] - groupBegin[pp]) * (uint32_t)coeffCount((int)pp) : 0u;
                S.jobPSlot[j] = (flags[r] & 2u) ? groupPool[pp + 1] + (pPos[r] - groupBegin[pp + 1]) * (uint32_t)coeffCount((int)pp + 1) : 0u;
                const float4 c = S.cell[node];
                JobDesc o;
                o.cx = c.x; o.cy = c.y; o.cz = c.z; o.half = c.w;
                o.hPos = hPos[r]; o.pPos = pPos[r]; o.src = S.slot[node];
                o.depth = S.depth[node]; o.degree = (uint8_t)pp; o.flags = flags[r]; o.pad = 0;
                S.jobsOut[k] = o;
            }
            if (chunk == 0 && tid == 0)
            {
                C.nOpen = sTotal[0]; C.nJobs = job0 + nSel; C.poolUsed = (uint32_t)poolNeed;
                C.roundJob0 = job0; C.roundJobs = nSel; C.jobsEvaluated += nSel; C.fitsEvaluated += nTasks;
            }
            __syncthreads();
        }
    }
}
