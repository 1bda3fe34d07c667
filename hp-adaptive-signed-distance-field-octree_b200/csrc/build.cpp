// build.cpp — Octree::Create on the GPU: batched greedy with exact replay.
//
// Reference (Source/HP/Octree.cpp): Create :312-352 → CreateRoot :792-801 → UniformlyRefine :112-191 →
// RunBuildThreadPool :194-309 (scheduler) + TickBuildThread :558-659 (worker: EstimateHImprovement :804-826,
// EstimatePImprovement :829-856, h/p decision :598-601) → ReallocCoeffs :474-555 → PerformContinuityPostProcess :1717-1762.
//
// The reference pops the max-error leaf, evaluates its refinement job (8 child fits + 1 p-fit) on a CPU thread, applies
// the better of the two and pushes the results back. A job's result is a pure function of (cell, degree, F), so here:
//   round r:  every leaf that has no cached job result is evaluated in ONE batch of fit kernels (fit_kernels.cuh);
//             only {raw error, c0} per fit come back to the host (16 B), coefficients stay in a device pool;
//   replay:   the host runs the reference's sequential scheduler on its priority queue (std::priority_queue with the
//             reference's predicate, so ties pop in the same order) using the cached results, with the reference's
//             totalCoeffError arithmetic, until it terminates or the top of the queue has no cached result → next round.
// This yields exactly the strict-greedy tree (the deterministic schedule the CPU checker defines: window 1, termination
// checked after every applied job; nearness weight from the exact cell mean, SURVEY.md F3-F5). Work computed for leaves
// that are never popped before termination is speculative waste, bounded by the number of final leaves.
#include <algorithm>
#include <functional>
#include <cmath>
#include <cstring>
#include <limits>
#include <mutex>
#include <queue>
#include <vector>
#include <cstdio>
#include <cstdlib>
#include "octree.h"
#include "comm.h"
#include "build_common.h"

namespace hpsdf
{
    namespace
    {
        struct Job
        {
            bool     coarse = false, doH = false, doP = false;
            uint32_t hSlot0 = 0, pSlot = 0;                  // pool slots: child c at hSlot0 + c * N_degree, the p-fit
            uint32_t hPos = 0, pPos = 0;                     // record indices of child 0 / the p-fit in their round
            double   hErr[8] = { 0 }, pErr = 0.0, hImp = 0.0, pImp = 0.0;
        };

        // JobDesc slots behind a round's job records that carry its RoundLayout to the device in the same copy
        constexpr size_t kLayoutSlots = (sizeof(RoundLayout) + sizeof(JobDesc) - 1) / sizeof(JobDesc);

        // Octree.h:95-102: max-heap on the error only
        struct QueuePredicate
        {
            bool operator()(const std::pair<uint64_t, double>& a, const std::pair<uint64_t, double>& b) const { return a.second < b.second; }
        };

        // Exact-mean limit of CalculatePolyWeighting / CalculateExpWeighting (Octree.cpp:1209-1247): the mean of the
        // approximant over its cell is coeffs[0] * NL[0][depth]^3 (orthonormal basis) instead of 100 std::rand() samples.
        double nearnessWeight(const hpsdf_config& cfg, double c0, uint32_t depth)
        {
            if (cfg.nearness_type == HPSDF_NEARNESS_NONE) return 1.0;
            const double nl = tables().nl[0][depth];
            double m = c0 * (nl * nl * nl);
            m = std::fabs(m);
            const double d = std::sqrt(3.0);
            if (cfg.nearness_type == HPSDF_NEARNESS_POLYNOMIAL)
            {
                const double k = std::pow(1.0 - m / d, cfg.nearness_strength);
                return std::min<double>(1.0, std::max<double>(k, 0.0));
            }
            return std::exp(-1.0 * cfg.nearness_strength * m / d);
        }

        class Builder
        {
        public:
            Builder(hpsdf_octree& t, const hpsdf_build_opts& o, const SdfProgramDev& prog)
                : t_(t), o_(o), prog_(prog), nodes_(t.nodes), cfg_(t.cfg) {}

            hpsdf_status run();

        private:
            hpsdf_octree&            t_;
            const hpsdf_build_opts&  o_;
            const SdfProgramDev&     prog_;
            std::vector<HostNode>&   nodes_;
            const hpsdf_config&      cfg_;
            cudaStream_t             stream_ = nullptr;
            bool                     ownStream_ = false;
            cudaEvent_t              ev0_ = nullptr, ev1_ = nullptr;

            struct Heap : std::priority_queue<std::pair<uint64_t, double>, std::vector<std::pair<uint64_t, double>>, QueuePredicate>
            {
                const std::vector<std::pair<uint64_t, double>>& entries() const { return c; }
            } queue_;
            // error histogram of the queue by binary exponent (bucket b holds errors in [2^(b-1101), 2^(b-1100)))
            static constexpr int kBuckets = 2200;
            std::vector<double>      bucketSum_ = std::vector<double>(kBuckets, 0.0);
            std::vector<uint32_t>    bucketCount_ = std::vector<uint32_t>(kBuckets, 0u);
            double                   applyLevel_ = std::numeric_limits<double>::infinity();   // entries >= this are certain to be popped
            size_t                   levelLogStart_ = 0;     // first apply-log entry of the current level
            double                   pendingMax_ = 0.0;      // largest error among pending_ (uncached) leaves
            std::vector<uint64_t>    evaluated_;
            std::vector<uint64_t>    coarseReady_;           // coarse cells whose degree-2 fit is cached
            std::vector<uint64_t>    ready_;                 // freshly evaluated leaves not yet in the heap
            bool                     levelTried_ = false;
            double                   evalLevel_ = 0.0;       // guaranteed level used to choose what to evaluate (also in strict mode)
            std::vector<int32_t>     jobOf_;        // per node: index into jobs_, -1 = no cached result
            std::vector<double>      errOf_;        // per node: its current (weighted) error
            std::vector<uint8_t>     inQueue_;      // per node: 1 while the leaf is in the priority queue
            std::vector<Job>         jobs_;
            // leaves of the conceptual queue whose job has not been evaluated yet, bucketed by error exponent like the
            // histogram, so that a round only touches the entries it selects (a flat list was rescanned every round:
            // 20 k entries x 18 rounds = a fifth of a C2 build)
            std::vector<std::vector<uint64_t>> pendB_ = std::vector<std::vector<uint64_t>>(kBuckets);
            size_t                   pendCount_ = 0;
            std::vector<uint64_t>    coarseCells_;  // the 16^3 cells in visiting order (UniformlyRefine)
            int                      pendTop_ = 0;  // no non-empty bucket above this one

            BuildWorkspace&          ws_ = t_.ctx->ws;
            DeviceBuf<double>&       pool_ = ws_.pool;  size_t poolUsed_ = 0;
            DeviceBuf<FitTask>&      dTasks_ = ws_.tasks;
            DeviceBuf<FitRecord>&    dRecs_ = ws_.recs;
            DeviceBuf<JobDesc>&      dJobs_ = ws_.jobs;
            PinnedBuf<JobDesc>&      hJobs_ = ws_.hJobs;
            PinnedBuf<FitRecord>&    hRecs_ = ws_.hRecs;

            double      total_ = 0.0;               // totalCoeffError, reference bookkeeping (Octree.cpp:212, 257, 272, 276)
            long double exactSum_ = 0.0L;
            long        unfitted_ = 0;
            int         rank_ = 0, world_ = 1;
            double      launchMs_ = 0.0;           // host time spent in upload / launch calls (diagnostics)
            size_t      strictSteps_ = 0, levelCalls_ = 0;   // diagnostics: strictly sequential pops; guaranteed-level computations
            ProgramSummary progSummary_;
            hpsdf_decision_log_entry lastApplied_{};      // last job applied before the termination cut
            double      lastTotal_ = 0.0, totalBeforeLast_ = 0.0;

            void         subdivide(uint64_t idx);
            void         refineUniform(uint64_t idx, uint32_t depth);
            hpsdf_status evaluateRound();
            bool         replay();                  // true = terminated
            hpsdf_status pack();
            void         logCutTies();
            void         applyJob(uint64_t idx, double err);
            void         computeLevel();
            static int   bucketOf(double e)
            {
                // binary exponent as frexp would give it for normal numbers, read from the bits (called ~10 times per job)
                if (!(e > 0.0)) return 0;
                uint64_t bits;
                memcpy(&bits, &e, 8);
                const int ex = (int)((bits >> 52) & 0x7FFu) - 1022;
                return std::min(std::max(ex + 1100, 0), kBuckets - 1);
            }
            // a new / changed leaf enters the conceptual queue: histogram + pending list (it reaches the heap once evaluated)
            void qPush(uint64_t idx, double err)
            {
                inQueue_[idx] = 1;
                const int b = bucketOf(err);
                bucketSum_[b] += err; bucketCount_[b]++;
                pendB_[b].push_back(idx);
                ++pendCount_;
                pendTop_ = std::max(pendTop_, b);
                pendingMax_ = std::max(pendingMax_, err);
            }
            void hPop()
            {
                const std::pair<uint64_t, double> t = queue_.top();
                queue_.pop();
                inQueue_[t.first] = 0;
                const int b = bucketOf(t.second);
                if (--bucketCount_[b] == 0) bucketSum_[b] = 0.0; else bucketSum_[b] -= t.second;
            }
            double conceptualTop() const
            {
                const double h = queue_.empty() ? 0.0 : queue_.top().second;
                return pendCount_ == 0 ? h : std::max(h, pendingMax_);
            }
            double checkValue() const
            {
                return o_.total_mode == HPSDF_TOTAL_EXACT_SUM
                     ? (unfitted_ > 0 ? std::numeric_limits<double>::infinity() : (double)exactSum_) : total_;
            }
        };

        // Subdivide (Octree.cpp:1115-1128)
        void Builder::subdivide(uint64_t idx)
        {
            nodes_[idx].child = nodes_.size();
            for (uint32_t i = 0; i < 8; ++i)
            {
                HostNode c;
                cornerAabb(nodes_[idx], i, c.mn, c.mx);
                c.depth = (uint8_t)(nodes_[idx].depth + 1);
                nodes_.push_back(c);
            }
        }

        // UniformlyRefine (Octree.cpp:112-191): pre-order DFS, Subdivide on first visit, children 0..7; the 16^3 cells at
        // depth 4 get degree 0 and enter the queue with err = 100 in visiting order.
        void Builder::refineUniform(uint64_t idx, uint32_t depth)
        {
            if (depth < (uint32_t)kCoarseDepth)
            {
                subdivide(idx);
                const uint64_t c = nodes_[idx].child;
                for (uint32_t i = 0; i < 8; ++i) refineUniform(c + i, depth + 1);
            }
            else
            {
                nodes_[idx].degree = 0;
                coarseCells_.push_back(idx);    // enters the queue with err = 100 in run(), in this (visiting) order
            }
        }

        // One batch: the refinement jobs of the pending (not yet evaluated) leaves at or above the evaluation level.
        hpsdf_status Builder::evaluateRound()
        {
            // ---- 1. which leaves: everything at or above the guaranteed level (computeLevel) is needed work; `speculate`
            //         octaves (factors of 8) below it are pre-evaluated so later levels find their results cached -------------
            if (o_.strict_order || applyLevel_ == std::numeric_limits<double>::infinity())
            {
                const double keep = applyLevel_;
                computeLevel();                 // refresh evalLevel_ for the current (sequential) state
                if (o_.strict_order || keep != std::numeric_limits<double>::infinity()) applyLevel_ = keep;
            }
            double level = std::min(evalLevel_, conceptualTop());
            for (uint32_t k = 0; k < o_.speculate; ++k) level *= 0.125;

            const double tTask0 = nowMs();
            // pass A: select, create the jobs, count fits per degree
            const size_t firstJob = jobs_.size();
            evaluated_.clear();
            uint32_t cnt[kMaxDegree + 2] = { 0 };
            // Everything at or above the level is needed work. If that is only a handful of jobs the round would cost a full
            // upload / launch / synchronise / replay cycle for them (10 of the 18 rounds of a C2 build selected fewer than 20
            // jobs), so the round is topped up to `min_round_jobs` with the next-largest pending errors: the greedy loop is
            // about to reach them anyway and their results stay cached until it does.
            // (not for mesh / octree programs by default: there a fit costs 10^3-10^4 BVH queries and speculation measured 25-35 % slower)
            const size_t minJobs = o_.min_round_jobs ? o_.min_round_jobs : (progSummary_.samplesExt ? 1u : 512u);
            const size_t pendBefore = pendCount_;
            auto select = [&](uint64_t idx) { evaluated_.push_back(idx); };
            const int levelBucket = bucketOf(level);
            pendingMax_ = 0.0;
            for (int b = pendTop_; b >= 0 && pendCount_ > 0; --b)
            {
                std::vector<uint64_t>& B = pendB_[b];
                if (B.empty()) { if (b == pendTop_ && pendTop_ > 0) --pendTop_; continue; }
                if (b < levelBucket && evaluated_.size() >= minJobs) break;
                size_t keep = 0;
                for (size_t k = 0; k < B.size(); ++k)
                {
                    const uint64_t idx = B[k];
                    if (errOf_[idx] >= level || evaluated_.size() < minJobs) select(idx);
                    else B[keep++] = idx;
                }
                pendCount_ -= B.size() - keep;
                B.resize(keep);
                if (keep) break;                 // the bucket was only partly taken: nothing below it is selected
            }
            while (pendTop_ > 0 && pendB_[pendTop_].empty()) --pendTop_;
            if (pendCount_) for (uint64_t idx : pendB_[pendTop_]) pendingMax_ = std::max(pendingMax_, errOf_[idx]);
            // several GPUs: every shard of a degree group gets the same mix of jobs (dealStride; only node numbering depends on
            // the order)
            if (world_ > 1 && evaluated_.size() > 2)
            {
                const size_t n = evaluated_.size();
                const size_t stride = dealStride((uint32_t)n);
                std::vector<uint64_t> perm(n);
                for (size_t k = 0; k < n; ++k) perm[k] = evaluated_[(k * stride) % n];
                evaluated_.swap(perm);
            }
            for (const uint64_t idx : evaluated_)
            {
                const HostNode& n = nodes_[idx];
                jobs_.emplace_back();
                Job& j = jobs_.back();
                j.coarse = std::abs(errOf_[idx] - kInitialErr) < std::numeric_limits<double>::epsilon() && n.degree == 0;   // Octree.cpp:806, 831
                if (j.coarse) { j.doP = true; cnt[kCoarseDegree]++; }
                else
                {
                    j.doH = n.depth < o_.max_depth;             // child fits at depth > TREE_MAX_DEPTH are never used (Octree.cpp:600-601)
                    j.doP = n.degree < o_.max_degree;           // nor is the p-fit of a max-degree node
                    if (j.doH) cnt[n.degree] += 8;
                    if (j.doP) cnt[n.degree + 1]++;
                }
                jobOf_[idx] = (int32_t)(jobs_.size() - 1);
            }
            static const bool dbgRounds = getenv("HPSDF_DEBUG_ROUNDS") != nullptr;
            if (dbgRounds) fprintf(stderr, "round %llu: pending %zu -> %zu, jobs %zu, heap %zu, level %.3e, passA %.3f ms\n", (unsigned long long)t_.stats.rounds,
                                   pendBefore, pendCount_, evaluated_.size(), queue_.entries().size(), level, nowMs() - tTask0);

            // task index == record index
            RoundLayout lay;
            uint64_t poolNeed = 0;
            const uint32_t nTasks = layoutRound(cnt, (uint32_t)poolUsed_, lay.groupBegin, lay.groupPool, poolNeed);
            if (poolNeed >= 0xFFFFFFF0ull) { setLastError("coefficient pool exceeds 2^32 doubles"); return HPSDF_ERR_OOM; }
            const size_t nJobs = evaluated_.size();
            HPSDF_CUDA(hJobs_.reserve(nJobs + kLayoutSlots));       // (pass B writes the records of a round without fits too)
            if (nTasks)
            {
                HPSDF_CUDA(pool_.reserve(poolNeed + 1024, stream_, poolUsed_));
                HPSDF_CUDA(dTasks_.reserve(nTasks));
                HPSDF_CUDA(dRecs_.reserve(nTasks));
                HPSDF_CUDA(hRecs_.reserve(nTasks));
                HPSDF_CUDA(dJobs_.reserve(nJobs + kLayoutSlots));
            }
            // pass B: one 32-byte job record per job straight into pinned memory; expandJobsDevKernel derives the fit tasks on
            // the device (the host used to write all 9 descriptors of a job: 75 k x 32 B per C2 build, a quarter of its time).
            uint32_t cursor[kMaxDegree + 2];
            for (int d = 0; d <= kMaxDegree + 1; ++d) cursor[d] = lay.groupBegin[d];
            auto slotOf = [&](int d, uint32_t pos) { return lay.groupPool[d] + (pos - lay.groupBegin[d]) * (uint32_t)coeffCount(d); };
            JobDesc* J = hJobs_.p;
            for (size_t k = 0; k < nJobs; ++k)
            {
                const uint64_t idx = evaluated_[k];
                const HostNode& n = nodes_[idx];
                Job& j = jobs_[firstJob + k];
                JobDesc& o = J[k];
                o.cx = (n.mn[0] + n.mx[0]) / 2.0f; o.cy = (n.mn[1] + n.mx[1]) / 2.0f; o.cz = (n.mn[2] + n.mx[2]) / 2.0f;   // AlignedBox::center() in f32
                o.half = (n.mx[0] - n.mn[0]) * 0.5f;
                o.depth = n.depth; o.degree = n.degree; o.pad = 0; o.src = n.slot; o.hPos = o.pPos = 0;
                if (j.coarse)                                                                    // Octree.cpp:840
                {
                    o.flags = 4u;
                    j.pPos = o.pPos = cursor[kCoarseDegree]++;
                    j.pSlot = slotOf(kCoarseDegree, j.pPos);
                    continue;
                }
                o.flags = (j.doH ? 1u : 0u) | (j.doP ? 2u : 0u);
                if (j.doH)                                                                       // Octree.cpp:820
                {
                    j.hPos = o.hPos = cursor[n.degree];
                    cursor[n.degree] += 8;
                    j.hSlot0 = slotOf(n.degree, j.hPos);
                }
                if (j.doP)                                                                       // Octree.cpp:846-851
                {
                    j.pPos = o.pPos = cursor[n.degree + 1]++;
                    j.pSlot = slotOf(n.degree + 1, j.pPos);
                }
            }
            poolUsed_ = poolNeed;
            t_.stats.host_tasks_ms += nowMs() - tTask0;

            // ---- 2. upload the job records with the layout behind them, expand, launch, read the fit records back ------------
            const double tLaunch0 = nowMs();
            if (nTasks)
            {
                memcpy(hJobs_.p + nJobs, &lay, sizeof(lay));
                HPSDF_CUDA(cudaMemcpyAsync(dJobs_.p, hJobs_.p, nJobs * sizeof(JobDesc) + sizeof(lay), cudaMemcpyHostToDevice, stream_));
                HPSDF_CUDA(launchExpandJobsDev(dJobs_.p, (uint32_t)nJobs, (const RoundLayout*)(dJobs_.p + nJobs), dTasks_.p, stream_));
                t_.stats.kernel_launches++;
                const hpsdf_status ls = launchRoundFits(t_, o_, prog_, progSummary_, stream_, cnt, lay, nTasks, rank_, world_, ev0_, ev1_);
                if (ls != HPSDF_OK) return ls;
                HPSDF_CUDA(cudaMemcpyAsync(hRecs_.p, dRecs_.p, nTasks * sizeof(FitRecord), cudaMemcpyDeviceToHost, stream_));
                const double tWait0 = nowMs();
                launchMs_ += tWait0 - tLaunch0;
                HPSDF_CUDA(cudaStreamSynchronize(stream_));
                t_.stats.device_wait_ms += nowMs() - tWait0;
                float ms = 0.0f;
                cudaEventElapsedTime(&ms, ev0_, ev1_);
                t_.stats.fit_kernel_ms += ms;
            }
            t_.stats.jobs_evaluated += jobs_.size() - firstJob;

            // ---- 3. errors (host, same expressions and libm as the CPU checker); the evaluated leaves enter the heap ------
            const double tRec0 = nowMs();
            const bool weighted = cfg_.nearness_type != HPSDF_NEARNESS_NONE;
            const FitRecord* R = hRecs_.p;
            for (size_t k = 0; k < nJobs && nTasks; ++k)
            {
                Job& j = jobs_[firstJob + k];
                const uint32_t depth = nodes_[evaluated_[k]].depth;
                auto err = [&](const FitRecord& r, uint32_t dep) { return weighted ? r.rawErr * nearnessWeight(cfg_, r.c0, dep) : r.rawErr; };
                if (j.coarse || j.doP) j.pErr = err(R[j.pPos], depth);
                if (j.doH) for (uint32_t c = 0; c < 8; ++c) j.hErr[c] = err(R[j.hPos + c], depth + 1);
            }
            for (size_t k = firstJob; k < jobs_.size(); ++k)
                if (jobs_[k].coarse) { jobs_[k].hImp = 0.0; jobs_[k].pImp = jobs_[k].pErr; }             // Octree.cpp:806-810, 836-843
            for (uint64_t idx : evaluated_)
            {
                if (jobs_[jobOf_[idx]].coarse) coarseReady_.push_back(idx);      // applied in the reference's pop order, see replay()
                else ready_.push_back(idx);                                       // enters the heap only if it is below the level
            }
            t_.stats.host_tasks_ms += nowMs() - tRec0;
            return HPSDF_OK;
        }

        // Guaranteed level. Take the queue in decreasing error order e1 >= e2 >= ...: entry k is certainly popped by the
        // strict greedy loop before it terminates if total - (e1 + ... + e_{k-1}) >= threshold, because popping an entry and
        // any of its descendants lowers the total by at most that entry's error. So is every descendant with a larger
        // error than e_k (the loop pops it before e_k). Entries at or above the level can therefore be applied in ANY
        // order without changing which leaves end up refined; only node numbering and the last bits of the running total
        // depend on the order. Computed from the per-exponent histogram, exact inside the bucket where the bound runs out.
        void Builder::computeLevel()
        {
            const double tSel0 = nowMs();
            const double inf = std::numeric_limits<double>::infinity();
            const double thr = cfg_.target_error_threshold;
            ++levelCalls_;
            levelLogStart_ = t_.applyLog.size();
            applyLevel_ = inf;
            double remaining = checkValue();
            evalLevel_ = conceptualTop();
            if (!(remaining >= thr) || (queue_.empty() && pendCount_ == 0)) { t_.stats.host_select_ms += nowMs() - tSel0; return; }
            int b = kBuckets - 1, crossing = -1;
            for (; b >= 0; --b)
            {
                if (!bucketCount_[b]) continue;
                const double after = remaining - bucketSum_[b] * (1.0 + 1e-9);
                if (after >= thr) { remaining = after; applyLevel_ = std::ldexp(0.5, b - 1100); continue; }   // whole bucket guaranteed
                crossing = b;
                break;
            }
            if (crossing >= 0)
            {
                std::vector<double> errs;
                for (const auto& e : queue_.entries()) if (bucketOf(e.second) == crossing) errs.push_back(e.second);
                for (uint64_t idx : pendB_[crossing]) errs.push_back(errOf_[idx]);
                std::sort(errs.begin(), errs.end(), std::greater<double>());
                size_t k = 0;
                for (; k < errs.size() && remaining >= thr; ++k) remaining -= errs[k] * (1.0 + 1e-9);
                // keep whole groups of equal errors together: never split a tie group out of order
                while (k > 0 && k < errs.size() && errs[k] == errs[k - 1]) --k;
                if (k > 0) applyLevel_ = errs[k - 1];
            }
            evalLevel_ = std::min(applyLevel_, evalLevel_);
            if (o_.strict_order) applyLevel_ = inf;          // strict mode: the level only steers what is evaluated
            t_.stats.host_select_ms += nowMs() - tSel0;
        }

        // One applied refinement: the body of the reference's output-drain loop (Octree.cpp:245-297) for a popped leaf.
        void Builder::applyJob(uint64_t idx, double err)
        {
            Job& j = jobs_[jobOf_[idx]];
            jobOf_[idx] = -1;
            const uint32_t p = nodes_[idx].degree, depth = nodes_[idx].depth;
            if (!j.coarse)
            {
                if (j.doH)
                {
                    double maxNew = 0.0;
                    for (int i = 0; i < 8; ++i) maxNew = std::max<double>(maxNew, j.hErr[i]);       // Octree.cpp:821
                    j.hImp = (1.0 / (7.0 * coeffCount(p))) * (err - 8.0 * maxNew);                  // Octree.cpp:825
                }
                if (j.doP) j.pImp = (1.0 / (coeffCount(p + 1) - coeffCount(p))) * (err - 8.0 * j.pErr);   // Octree.cpp:854
            }
            // Octree.cpp:600-601 with BASIS_MAX_DEGREE-1 -> max_degree, TREE_MAX_DEPTH -> max_depth. A coarse cell always
            // takes its degree-2 fit (the reference is undefined if that fit's error is exactly 0, SURVEY.md App. C).
            const bool refineP = j.coarse || (p < o_.max_degree && (depth == o_.max_depth || j.pImp > j.hImp));
            const bool refineH = depth < o_.max_depth && !refineP;

            if (!j.coarse && j.doH && j.doP)
            {
                const double mag = std::max(std::fabs(j.pImp), std::fabs(j.hImp));
                const double margin = mag > 0.0 ? std::fabs(j.pImp - j.hImp) / mag : 0.0;
                if (margin <= 1e-9)
                {
                    hpsdf_decision_log_entry e{};
                    e.node_idx = idx; e.depth = depth; e.degree = p; e.chose_p = refineP; e.kind = 0;
                    for (int a = 0; a < 3; ++a) e.centre[a] = (nodes_[idx].mn[a] + nodes_[idx].mx[a]) / 2.0f;
                    e.p_improvement = j.pImp; e.h_improvement = j.hImp; e.relative_margin = margin;
                    t_.decisionLog.push_back(e);
                    t_.stats.near_tie_decisions++;
                }
            }

            if (refineP)
            {
                total_ += (j.pErr - err);                                                            // Octree.cpp:257
                if (j.coarse) unfitted_--; else exactSum_ -= (long double)err;
                exactSum_ += (long double)j.pErr;
                nodes_[idx].slot   = j.pSlot;                                                        // Octree.cpp:286
                nodes_[idx].degree = (uint8_t)(j.coarse ? kCoarseDegree : p + 1);
                errOf_[idx] = j.pErr;
                qPush(idx, j.pErr);                                                                  // Octree.cpp:289-290
                t_.stats.jobs_applied_p++;
                t_.applyLog.push_back({ idx, 0u, p, err, j.pErr, j.pImp, j.hImp, checkValue() });
            }
            else if (refineH)
            {
                nodes_[idx].degree = kInternalTag;                                                   // Octree.cpp:265-272
                subdivide(idx);
                total_ -= err;
                exactSum_ -= (long double)err;
                jobOf_.resize(nodes_.size(), -1);
                errOf_.resize(nodes_.size(), 0.0);
                inQueue_.resize(nodes_.size(), 0);
                double mx = 0.0;
                for (uint32_t i = 0; i < 8; ++i)
                {
                    const uint64_t c = nodes_[idx].child + i;                                        // Octree.cpp:275-290
                    total_ += j.hErr[i];
                    exactSum_ += (long double)j.hErr[i];
                    nodes_[c].slot = j.hSlot0 + i * (uint32_t)coeffCount((int)p);
                    nodes_[c].degree = (uint8_t)p;
                    errOf_[c] = j.hErr[i];
                    qPush(c, j.hErr[i]);
                    mx = std::max(mx, j.hErr[i]);
                }
                t_.stats.jobs_applied_h++;
                t_.applyLog.push_back({ idx, 1u, p, err, mx, j.pImp, j.hImp, checkValue() });
            }
            // else: degree and depth both at their maximum — the node leaves the queue (Octree.cpp:643-655)

            if (refineP || refineH)
            {
                lastApplied_.node_idx = idx; lastApplied_.depth = depth; lastApplied_.degree = p; lastApplied_.chose_p = refineP;
                lastApplied_.kind = 1; lastApplied_.p_improvement = j.pImp; lastApplied_.h_improvement = j.hImp;
                for (int a = 0; a < 3; ++a) lastApplied_.centre[a] = (nodes_[idx].mn[a] + nodes_[idx].mx[a]) / 2.0f;
                totalBeforeLast_ = lastTotal_; lastTotal_ = checkValue();
            }
            if (cfg_.enable_logging)                                                                 // Octree.cpp:292-296
                printf("\n%.11f\t%zu\t%f, %f, %f", total_, nodes_.size(), (double)(nodes_[idx].mn[0] + nodes_[idx].mx[0]) / 2.0,
                       (double)(nodes_[idx].mn[1] + nodes_[idx].mx[1]) / 2.0, (double)(nodes_[idx].mn[2] + nodes_[idx].mx[2]) / 2.0);
        }

        // The reference's scheduler loop (Octree.cpp:213-302) driven by cached job results. The heap holds only leaves whose
        // job is cached; leaves still waiting for a batch sit in pending_ (pendingMax_ = their largest error), so the
        // conceptual queue of the reference = heap + pending. Entries at or above the guaranteed level are applied as soon
        // as they are cached; below the level the loop is the strict one: termination check, then pop the overall maximum
        // if it is cached. Every time the strict part is reached the state is one the sequential greedy loop passes through.
        bool Builder::replay()
        {
            const double thr = cfg_.target_error_threshold;
            const double inf = std::numeric_limits<double>::infinity();
            bool done = false;
            levelTried_ = false;
            if (!coarseReady_.empty())
            {
                // visiting order of UniformlyRefine = ascending node index (pre-order allocation); a multi-GPU round deals its jobs out
                std::sort(coarseReady_.begin(), coarseReady_.end());
                // Coarse stage (Octree.cpp:112-191, 228-238): all 16^3 cells sit in the reference's queue with err = 100; each is
                // popped, fitted and pushed back with its real error. The ORDER in which the equal keys pop is a property of
                // the heap algorithm and of the re-pushed entries, and it matters: totalCoeffError starts at 8^4 * 100, so
                // the first errors added are rounded at ulp(4e5) = 5.8e-11 and the running total depends on the order at
                // the 1e-9 level (SURVEY.md F4). Replay the same push/pop sequence on a scratch std::priority_queue.
                std::priority_queue<std::pair<uint64_t, double>, std::vector<std::pair<uint64_t, double>>, QueuePredicate> sim;
                for (uint64_t idx : coarseReady_) sim.push({ idx, kInitialErr });                         // visiting order, Octree.cpp:176-177
                std::vector<uint64_t> order;
                order.reserve(coarseReady_.size());
                for (size_t k = 0; k < coarseReady_.size(); ++k)
                {
                    const std::pair<uint64_t, double> top = sim.top();
                    sim.pop();
                    order.push_back(top.first);
                    sim.push({ top.first, jobs_[jobOf_[top.first]].pErr });
                }
                for (uint64_t idx : order)
                {
                    inQueue_[idx] = 0;
                    const int b = bucketOf(kInitialErr);
                    if (--bucketCount_[b] == 0) bucketSum_[b] = 0.0; else bucketSum_[b] -= kInitialErr;
                    applyJob(idx, kInitialErr);
                }
                coarseReady_.clear();
                applyLevel_ = inf;
            }
            // freshly evaluated leaves at or above the level need no ordering at all: apply them directly; the rest go to the heap
            for (size_t k = 0; k < ready_.size(); ++k)
            {
                const uint64_t idx = ready_[k];
                const double err = errOf_[idx];
                if (err >= applyLevel_)
                {
                    inQueue_[idx] = 0;
                    const int b = bucketOf(err);
                    if (--bucketCount_[b] == 0) bucketSum_[b] = 0.0; else bucketSum_[b] -= err;
                    applyJob(idx, err);
                }
                else queue_.push({ idx, err });
            }
            ready_.clear();
            for (;;)
            {
                if (queue_.empty() && pendCount_ == 0) { done = true; break; }                          // nodeQueue.empty(), Octree.cpp:216
                if (!queue_.empty() && queue_.top().second >= applyLevel_)
                {
                    const std::pair<uint64_t, double> top = queue_.top();
                    hPop();
                    applyJob(top.first, top.second);
                    continue;
                }
                if (pendingMax_ >= applyLevel_ && pendCount_ != 0) break;     // entries above the level still wait for their results
                if (checkValue() < thr) { done = true; break; }                                          // Octree.cpp:216
                if (!queue_.empty() && (pendCount_ == 0 || queue_.top().second >= pendingMax_))
                {
                    const std::pair<uint64_t, double> top = queue_.top();                                // Octree.cpp:231: the overall maximum
                    hPop();
                    applyJob(top.first, top.second);          // strict step; the state after it is a sequential-greedy state
                    ++strictSteps_;
                    applyLevel_ = inf;                        // a level is only valid for the state it was computed in
                    levelTried_ = false;
                    continue;
                }
                // the overall maximum has no cached result. This is a sequential-greedy state: find the level down to which
                // entries are certain to be popped, so the loop can go on past it (once per state)
                if (!o_.strict_order && applyLevel_ == inf && !levelTried_)
                {
                    computeLevel();
                    levelTried_ = true;
                    if (!queue_.empty() && queue_.top().second >= applyLevel_) continue;
                }
                break;
            }
            return done;
        }

        void Builder::logCutTies()
        {
            logCutTieGroup(t_, errOf_, levelLogStart_, queue_.empty() && pendCount_ == 0);
        }

        // ReallocCoeffs (Octree.cpp:474-555): DFS from the root's children by child slot; leaves packed in visiting order.
        hpsdf_status Builder::pack()
        {
            return packCoefficients(t_, pool_.p, stream_);
        }

        hpsdf_status Builder::run()
        {
            const double t0 = nowMs();
            std::lock_guard<std::mutex> wsLock(*(std::mutex*)t_.ctx->wsMutex);
            stream_ = o_.stream ? (cudaStream_t)o_.stream : ws_.stream;
            ev0_ = ws_.ev0; ev1_ = ws_.ev1;
            if (o_.comm) { rank_ = commRank(o_.comm); world_ = commWorld(o_.comm); }
            progSummary_ = summarizeProgram(prog_);
            t_.stats.sdf_flops_per_eval = progSummary_.flopsPerEval;

            hpsdf_status st = HPSDF_OK;
            const double tSetup0 = nowMs();
            // CreateRoot (Octree.cpp:792-801) + UniformlyRefine
            nodes_.clear();
            // growth of these vectors during the replay is pure overhead: start from the size of the last build on this device
            const size_t guess = std::max<size_t>(ws_.lastNodeCount + ws_.lastNodeCount / 4, 8192);
            nodes_.reserve(guess);
            errOf_.reserve(guess); jobOf_.reserve(guess); inQueue_.reserve(guess);
            jobs_.reserve(guess / 2);
            t_.applyLog.reserve(guess / 2);
            HostNode root;
            root.depth = 0;
            for (int i = 0; i < 3; ++i) { root.mn[i] = -0.5f; root.mx[i] = 0.5f; }
            nodes_.push_back(root);
            subdivide(0);
            for (uint32_t i = 0; i < 8; ++i) refineUniform(1 + i, 1);
            errOf_.assign(nodes_.size(), kInitialErr);
            jobOf_.assign(nodes_.size(), -1);
            inQueue_.assign(nodes_.size(), 0);
            for (uint64_t idx : coarseCells_) qPush(idx, kInitialErr);                                  // Octree.cpp:176-177
            total_ = std::pow(8, 4) * kInitialErr;                                                      // Octree.cpp:212
            unfitted_ = (long)pendCount_;
            lastTotal_ = totalBeforeLast_ = total_;
            computeLevel();
            if (getenv("HPSDF_DEBUG_ROUNDS")) fprintf(stderr, "setup %.3f ms\n", nowMs() - tSetup0);

            double replayMs = 0.0;
            size_t stallGuard = 0;
            for (;;)
            {
                st = evaluateRound();
                if (st != HPSDF_OK) break;
                const double r0 = nowMs();
                const bool done = replay();
                replayMs += nowMs() - r0;
                if (done) break;
                if (pendCount_ == 0) { setLastError("internal: replay stalled with nothing to evaluate"); st = HPSDF_ERR_CUDA; break; }
                if (++stallGuard > 100000) { setLastError("internal: build does not converge"); st = HPSDF_ERR_CUDA; break; }
            }
            if (getenv("HPSDF_DEBUG_ROUNDS")) fprintf(stderr, "launch calls %.3f ms, strict steps %zu, level computations %zu, applied %zu\n", launchMs_, strictSteps_, levelCalls_, t_.applyLog.size());
            const double tPack0 = nowMs();
            if (st == HPSDF_OK) st = pack();
            t_.stats.pack_ms = nowMs() - tPack0;
            if (st == HPSDF_OK)
            {
                t_.stats.total_error = o_.total_mode == HPSDF_TOTAL_EXACT_SUM ? (double)exactSum_ : total_;
                t_.stats.exact_total_error = (double)exactSum_;
                const double thr = cfg_.target_error_threshold;
                t_.stats.cut_margin = (thr - checkValue()) / thr;
                if (lastApplied_.kind == 1)
                {
                    // how far above the threshold the total was before the last applied job, relative to the threshold
                    lastApplied_.relative_margin = std::min(std::fabs(totalBeforeLast_ - thr), std::fabs(thr - checkValue())) / thr;
                    t_.decisionLog.push_back(lastApplied_);
                }
                logCutTies();
                t_.stats.host_replay_ms = replayMs;
                if (cfg_.continuity_enforce)
                {
                    const double c0 = nowMs();
                    st = continuityPostProcess(t_, o_, stream_);                                          // Octree.cpp:341-344
                    t_.stats.continuity_ms = nowMs() - c0;
                }
            }
            const double tFin0 = nowMs();
            if (st == HPSDF_OK) st = finalizeQueryStructures(t_, stream_);
            t_.stats.finalize_ms = nowMs() - tFin0;
            if (st == HPSDF_OK)
            {
                uint64_t leaves = 0;
                for (const HostNode& n : nodes_) leaves += n.child == kNoChild;
                t_.stats.n_nodes = nodes_.size(); ws_.lastNodeCount = nodes_.size(); t_.stats.n_leaves = leaves; t_.stats.n_coeffs = t_.nCoeffs;
            }
            cudaStreamSynchronize(stream_);
            t_.stats.total_ms = nowMs() - t0;
            return st;
        }
    }

    // Octree::Create with the greedy loop replayed on the host (hpsdf_build_opts.scheduler = 1, or strict_order): the round-1
    // implementation, kept as the cross-check of the device-resident scheduler (build_device.cpp) and for strict node numbering.
    hpsdf_status buildOctreeHost(hpsdf_octree& t, const hpsdf_build_opts& opts, const SdfProgramDev& prog)
    {
        Builder b(t, opts, prog);
        return b.run();
    }
}
