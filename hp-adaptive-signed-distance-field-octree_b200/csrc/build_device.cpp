// build_device.cpp — Octree::Create with the greedy loop resident on the device: host driver of sched_kernels.cuh.
//
// Reference (Source/HP/Octree.cpp): Create :312-352 -> CreateRoot :792-801 -> UniformlyRefine :112-191 -> RunBuildThreadPool
// :194-309 + TickBuildThread :558-659 -> ReallocCoeffs :474-555 -> PerformContinuityPostProcess :1717-1762.
//
// Per round the host does three things: read the 112-byte header the scheduler kernel wrote into mapped pinned memory (how
// many fits of which degree the next round has), launch expandJobsDevKernel + the round's fits (launchRoundFits in
// build_common.cpp: one fit kernel per degree present + the NCCL exchange when the round is sharded over several GPUs), and
// launch the scheduler kernel again. Queue, decision, error bookkeeping, node allocation and job selection never leave the
// device; at the end the node arrays come back once.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <queue>
#include <vector>
#include "octree.h"
#include "comm.h"
#include "sched.h"
#include "build_common.h"

namespace hpsdf
{
    cudaError_t launchSchedRound(const SchedDev& S, const uint16_t* coarseOrder, cudaStream_t stream);                    // kernels.cu
    struct FinishHeader { volatile uint32_t seq; uint32_t nLeaves, nCoeffs, nCoeffsPad; SchedCounters counters; };     // finish_kernels.cuh
    void        printMeshStats();                                                                                         // fit_kernels.cuh
    cudaError_t launchSchedIngest(const SchedDev& S, uint32_t nJobs, cudaStream_t stream);
    cudaError_t launchSchedSelect(const SchedDev& S, uint32_t openEstimate, cudaStream_t stream);
    cudaError_t launchSchedInit(const SchedDev& S, const SchedTemplates& T, const SchedCounters& c0, const RoundLayout& lay, cudaStream_t stream);
    size_t      finishSortTempBytes(uint32_t capNodes);
    cudaError_t launchFinishOrder(const SchedDev& S, uint32_t nNodes, uint32_t* keys, uint32_t* vals, uint32_t* keysAlt, uint32_t* valsAlt,
                                  uint32_t* counter, void* tmp, size_t tmpBytes, uint32_t* cstartOf, uint32_t* padOf, FinishHeader* hdr, uint32_t seq,
                                  cudaStream_t stream);
    cudaError_t launchEmitTree(const SchedDev& S, uint32_t nNodes, const uint32_t* cstartOf, const uint32_t* padOf, const double* pool,
                               double* packed, QNode* qnodes, unsigned char* image, cudaStream_t stream);
    cudaError_t launchPadCoefficients(const SchedDev& S, uint32_t nNodes, const uint32_t* cstartOf, const uint32_t* padOf, const double* packed,
                                      double* padded, cudaStream_t stream);

    namespace
    {
        constexpr uint32_t kCoarseCells = 4096, kCoarseNodes = 4681;

        // Pop order of the 16^3 coarse cells from the reference's std::priority_queue (Octree.cpp:176-177, 228-238): all keys
        // start at 100 and every popped cell is pushed back with its real error (< 100). Each comparison the heap makes has
        // an outcome that does not depend on those errors as far as the unfitted entries are concerned (100 against 100, 100
        // against a smaller key, or two re-pushed keys whose exchange moves no unfitted entry), so the order is a constant of
        // libstdc++'s push_heap / pop_heap: derived once by running them on dummy keys.
        std::vector<uint16_t> coarsePopOrder()
        {
            struct Pred { bool operator()(const std::pair<uint32_t, double>& a, const std::pair<uint32_t, double>& b) const { return a.second < b.second; } };
            std::priority_queue<std::pair<uint32_t, double>, std::vector<std::pair<uint32_t, double>>, Pred> q;
            for (uint32_t i = 0; i < kCoarseCells; ++i) q.push({ i, kInitialErr });
            std::vector<uint16_t> order;
            order.reserve(kCoarseCells);
            for (uint32_t k = 0; k < kCoarseCells; ++k)
            {
                const std::pair<uint32_t, double> top = q.top();
                q.pop();
                order.push_back((uint16_t)top.first);
                q.push({ top.first, 1e-6 / (1.0 + top.first) });
            }
            return order;
        }

        // Device arrays of one build, owned by the device context (one build at a time per device).
        struct SchedWorkspace
        {
            uint32_t  cap = 0;                   // nodes = jobs = log entries
            char*     arena = nullptr;
            SchedDev  dev{};
            RoundHeader* hostHdr = nullptr;      // mapped pinned
            RoundHeader* devHdr = nullptr;
            // templates of the uniform depth-4 start (UniformlyRefine, Octree.cpp:112-191)
            char*     tmpl = nullptr;
            float4*   tCell = nullptr; uint32_t* tChild = nullptr; uint32_t* tCode = nullptr; uint8_t* tDepth = nullptr; uint8_t* tDegree = nullptr; uint8_t* tState = nullptr;
            uint32_t* tJobNode = nullptr; uint32_t* tJobPSlot = nullptr; uint32_t* tJobPPos = nullptr; uint8_t* tJobFlags = nullptr;
            JobDesc*  tJobs = nullptr;
            uint16_t* coarseOrder = nullptr;
            uint32_t* tTop = nullptr;            // 16^3 entry table of the Query kernel (fixed by the uniform start)
            SchedTemplates tpl{};
            // finish: DFS order of the leaves
            uint32_t* sortKeys = nullptr; uint32_t* sortVals = nullptr; uint32_t* sortKeysAlt = nullptr; uint32_t* sortValsAlt = nullptr;
            uint32_t* cstartOf = nullptr; uint32_t* padOf = nullptr; uint32_t* leafCounter = nullptr;
            void*     sortTmp = nullptr; size_t sortTmpBytes = 0;
            FinishHeader* hostFin = nullptr; FinishHeader* devFin = nullptr;
            uint32_t  finSeq = 0;
            std::vector<cudaEvent_t> ev;         // pairs around the fit launches of a round
            std::vector<cudaEvent_t> dbgEv;      // HPSDF_DEBUG_ROUNDS=2: one more per round, after the exchange
            // pinned staging for the final read-back
            PinnedBuf<char> hBack;
        };

        size_t alignUp(size_t b) { return (b + 255) & ~(size_t)255; }

        hpsdf_status ensureTemplates(SchedWorkspace& w)
        {
            if (w.tmpl) return HPSDF_OK;
            std::vector<float4> cell(kCoarseNodes);
            std::vector<uint32_t> child(kCoarseNodes, kNone), code(kCoarseNodes, 0);
            std::vector<uint8_t> depth(kCoarseNodes, 0), degree(kCoarseNodes, kInternalTag), state(kCoarseNodes, kStInternal);
            std::vector<uint32_t> jobNode; jobNode.reserve(kCoarseCells);
            uint32_t next = 1;
            cell[0] = make_float4(0.0f, 0.0f, 0.0f, 0.5f);
            // pre-order: Subdivide on first visit (8 consecutive nodes at the end), then the children 0..7
            struct Rec
            {
                std::vector<float4>& cell; std::vector<uint32_t>& child; std::vector<uint32_t>& code; std::vector<uint8_t>& depth;
                std::vector<uint8_t>& degree; std::vector<uint8_t>& state; std::vector<uint32_t>& jobNode; uint32_t& next;
                void visit(uint32_t idx, uint32_t d)
                {
                    if (d < (uint32_t)kCoarseDepth)
                    {
                        child[idx] = next;
                        const float4 pc = cell[idx];
                        const float q = pc.w * 0.5f;
                        for (uint32_t c = 0; c < 8; ++c)
                        {
                            const uint32_t k = next + c;
                            cell[k] = make_float4(pc.x + ((c & 1u) ? q : -q), pc.y + ((c & 2u) ? q : -q), pc.z + ((c & 4u) ? q : -q), q);
                            depth[k] = (uint8_t)(d + 1);
                            code[k] = code[idx] | (c << (27 - 3 * (int)d));
                        }
                        const uint32_t c0 = next;
                        next += 8;
                        for (uint32_t c = 0; c < 8; ++c) visit(c0 + c, d + 1);
                    }
                    else
                    {
                        degree[idx] = 0; state[idx] = kStEval;
                        jobNode.push_back(idx);
                    }
                }
            } rec{ cell, child, code, depth, degree, state, jobNode, next };
            rec.visit(0, 0);
            if (next != kCoarseNodes || jobNode.size() != kCoarseCells) { setLastError("internal: uniform start template"); return HPSDF_ERR_CUDA; }
            std::vector<uint32_t> jobPSlot(kCoarseCells), jobPPos(kCoarseCells);
            std::vector<uint8_t> jobFlags(kCoarseCells, 2u);
            std::vector<JobDesc> jobs(kCoarseCells);
            for (uint32_t j = 0; j < kCoarseCells; ++j)
            {
                jobPSlot[j] = j * (uint32_t)coeffCount(kCoarseDegree); jobPPos[j] = j;
                const float4 c = cell[jobNode[j]];
                JobDesc& o = jobs[j];
                o.cx = c.x; o.cy = c.y; o.cz = c.z; o.half = c.w; o.hPos = 0; o.pPos = j; o.src = 0;
                o.depth = (uint8_t)kCoarseDepth; o.degree = 0; o.flags = 4u; o.pad = 0;
            }
            const std::vector<uint16_t> order = coarsePopOrder();
            // depth-4 entry table: node of cell (ix, iy, iz) of the 16^3 grid at index ix + 16 iy + 256 iz
            std::vector<uint32_t> top(4096);
            for (uint32_t codeIdx = 0; codeIdx < 4096; ++codeIdx)
            {
                const uint32_t ix = codeIdx & 15, iy = (codeIdx >> 4) & 15, iz = codeIdx >> 8;
                uint32_t cur = 0;
                for (int l = 3; l >= 0; --l) cur = child[cur] + ((ix >> l) & 1) + 2 * ((iy >> l) & 1) + 4 * ((iz >> l) & 1);
                top[codeIdx] = cur;
            }
            const size_t bytes = alignUp(4096 * 4) + alignUp(kCoarseNodes * 16) + 2 * alignUp(kCoarseNodes * 4) + 3 * alignUp(kCoarseNodes) + 3 * alignUp(kCoarseCells * 4) +
                                 alignUp(kCoarseCells) + alignUp(kCoarseCells * sizeof(JobDesc)) + alignUp(kCoarseCells * 2);
            HPSDF_CUDA(cudaMalloc((void**)&w.tmpl, bytes));
            char* p = w.tmpl;
            auto put = [&](const void* src, size_t n) { char* at = p; cudaMemcpy(at, src, n, cudaMemcpyHostToDevice); p += alignUp(n); return at; };
            w.tCell = (float4*)put(cell.data(), kCoarseNodes * 16);
            w.tChild = (uint32_t*)put(child.data(), kCoarseNodes * 4);
            w.tCode = (uint32_t*)put(code.data(), kCoarseNodes * 4);
            w.tDepth = (uint8_t*)put(depth.data(), kCoarseNodes);
            w.tDegree = (uint8_t*)put(degree.data(), kCoarseNodes);
            w.tState = (uint8_t*)put(state.data(), kCoarseNodes);
            w.tJobNode = (uint32_t*)put(jobNode.data(), kCoarseCells * 4);
            w.tJobPSlot = (uint32_t*)put(jobPSlot.data(), kCoarseCells * 4);
            w.tJobPPos = (uint32_t*)put(jobPPos.data(), kCoarseCells * 4);
            w.tJobFlags = (uint8_t*)put(jobFlags.data(), kCoarseCells);
            w.tJobs = (JobDesc*)put(jobs.data(), kCoarseCells * sizeof(JobDesc));
            w.coarseOrder = (uint16_t*)put(order.data(), kCoarseCells * 2);
            w.tTop = (uint32_t*)put(top.data(), 4096 * 4);
            HPSDF_CUDA(cudaHostAlloc((void**)&w.hostHdr, sizeof(RoundHeader) + 64 + sizeof(FinishHeader) + 64, cudaHostAllocMapped));
            HPSDF_CUDA(cudaHostGetDevicePointer((void**)&w.devHdr, w.hostHdr, 0));
            memset((void*)w.hostHdr, 0, sizeof(RoundHeader) + 64 + sizeof(FinishHeader) + 64);
            w.tpl.cell = w.tCell; w.tpl.child = w.tChild; w.tpl.code = w.tCode; w.tpl.depth = w.tDepth; w.tpl.degree = w.tDegree; w.tpl.state = w.tState;
            w.tpl.jobNode = w.tJobNode; w.tpl.jobPSlot = w.tJobPSlot; w.tpl.jobPPos = w.tJobPPos; w.tpl.jobFlags = w.tJobFlags;
            w.tpl.nNodes = kCoarseNodes; w.tpl.nJobs = kCoarseCells;
            w.hostFin = (FinishHeader*)((char*)w.hostHdr + sizeof(RoundHeader) + 64);
            w.devFin = (FinishHeader*)((char*)w.devHdr + sizeof(RoundHeader) + 64);
            return HPSDF_OK;
        }

        hpsdf_status ensureCapacity(SchedWorkspace& w, uint32_t cap)
        {
            if (w.cap >= cap) return HPSDF_OK;
            if (w.arena) { cudaFree(w.arena); w.arena = nullptr; w.cap = 0; }
            const size_t n = cap;
            const size_t sizes[] = {
                n * 16, n * 4, n * 4, n * 8, n * 4, n * 4, n, n, n,                 // nodes: cell child slot err code jobOf depth degree state
                n * 4, n * 4, n * 4, n * 4, n * 4, n * 72, n,                        // jobs: node hslot pslot hpos ppos err flags
                n * 4, n * 4, 2 * n * 4, n * 4, (n / kSelChunk + 2) * 64,           // open, cached, scratch, second open list, chunk counters
                (size_t)kSubBuckets * 4, (size_t)kSubBuckets * 8, (size_t)kSubBuckets * 4,
                n * sizeof(JobDesc), sizeof(RoundLayout), n * sizeof(hpsdf_apply_log_entry), 4096 * sizeof(hpsdf_decision_log_entry),
                sizeof(SchedCounters),
                n * 4, n * 4, n * 4, n * 4, n * 4, n * 4, 256, finishSortTempBytes(cap) };   // finish: sort keys / values (x2), cstart, padded start, leaf counter, CUB temp
            size_t total = 0;
            for (size_t s : sizes) total += alignUp(s);
            cudaError_t e = cudaMalloc((void**)&w.arena, total);
            if (e != cudaSuccess) return failCuda(e, "scheduler workspace");
            char* p = w.arena;
            int k = 0;
            auto take = [&]() { char* at = p; p += alignUp(sizes[k++]); return (void*)at; };
            SchedDev& d = w.dev;
            d.cell = (float4*)take(); d.child = (uint32_t*)take(); d.slot = (uint32_t*)take(); d.err = (double*)take(); d.code = (uint32_t*)take();
            d.jobOf = (uint32_t*)take(); d.depth = (uint8_t*)take(); d.degree = (uint8_t*)take(); d.state = (uint8_t*)take();
            d.jobNode = (uint32_t*)take(); d.jobHSlot = (uint32_t*)take(); d.jobPSlot = (uint32_t*)take(); d.jobHPos = (uint32_t*)take();
            d.jobPPos = (uint32_t*)take(); d.jobErr = (double*)take(); d.jobFlags = (uint8_t*)take();
            d.open = (uint32_t*)take(); d.cached = (uint32_t*)take(); d.scratch = (uint32_t*)take(); d.openAlt = (uint32_t*)take();
            d.chunkCounts = (uint32_t*)take();
            d.allCnt = (uint32_t*)take(); d.allSum = (unsigned long long*)take(); d.pendCnt = (uint32_t*)take();
            d.jobsOut = (JobDesc*)take(); d.layout = (RoundLayout*)take(); d.log = (hpsdf_apply_log_entry*)take();
            d.decisions = (hpsdf_decision_log_entry*)take(); d.ctr = (SchedCounters*)take();
            w.sortKeys = (uint32_t*)take(); w.sortVals = (uint32_t*)take(); w.sortKeysAlt = (uint32_t*)take(); w.sortValsAlt = (uint32_t*)take();
            w.cstartOf = (uint32_t*)take(); w.padOf = (uint32_t*)take(); w.leafCounter = (uint32_t*)take();
            w.sortTmpBytes = sizes[k]; w.sortTmp = take();
            d.capNodes = cap; d.capJobs = cap; d.capLog = cap; d.capDecisions = 4096;
            w.cap = cap;
            return HPSDF_OK;
        }

        class DeviceBuilder
        {
        public:
            DeviceBuilder(hpsdf_octree& t, const hpsdf_build_opts& o, const SdfProgramDev& prog) : t_(t), o_(o), prog_(prog), ws_(t.ctx->ws) {}
            hpsdf_status run(bool& fallBack);

        private:
            hpsdf_octree&           t_;
            const hpsdf_build_opts& o_;
            const SdfProgramDev&    prog_;
            BuildWorkspace&         ws_;
            cudaStream_t            stream_ = nullptr;
            int                     rank_ = 0, world_ = 1;
            ProgramSummary          progSummary_;
            double                  fitMs_ = 0.0;
            size_t                  evUsed_ = 0;
            uint32_t                nNodesFinal_ = 0;

            hpsdf_status launchRound(SchedWorkspace& w, const uint32_t* cnt, const RoundLayout& lay, uint32_t nTasks);
            hpsdf_status waitHeader(SchedWorkspace& w, uint32_t seq);
            hpsdf_status attempt(SchedWorkspace& w, uint32_t& doneCode);
            hpsdf_status finish(SchedWorkspace& w);
        };

        hpsdf_status DeviceBuilder::waitHeader(SchedWorkspace& w, uint32_t seq)
        {
            // the kernel writes the header into mapped host memory and publishes it with `seq`; polling it costs ~2 us where
            // a stream synchronisation costs 10+. The stream is queried from time to time so that a failed launch cannot hang us.
            const double t0 = nowMs();
            for (uint64_t spin = 0;; ++spin)
            {
                if (w.hostHdr->seq == seq) break;
                if ((spin & 0xFFF) == 0xFFF)
                {
                    if (nowMs() - t0 > 120000.0) { setLastError("internal: scheduler kernel did not answer within 120 s"); return HPSDF_ERR_CUDA; }
                    const cudaError_t q = cudaStreamQuery(stream_);
                    if (q != cudaSuccess && q != cudaErrorNotReady) return failCuda(q, "scheduler kernel");
                    if (q == cudaSuccess && w.hostHdr->seq != seq)
                    {
                        // the stream drained: give the write a last chance to become visible, then give up
                        cudaStreamSynchronize(stream_);
                        if (w.hostHdr->seq == seq) break;
                        setLastError("internal: scheduler kernel finished without publishing its header");
                        return HPSDF_ERR_CUDA;
                    }
                }
            }
            std::atomic_thread_fence(std::memory_order_acquire);
            t_.stats.device_wait_ms += nowMs() - t0;
            return HPSDF_OK;
        }

        // The fit launches of one round between the next pair of the workspace's events (HPSDF_DEBUG_ROUNDS=2: one more after
        // the exchange).
        hpsdf_status DeviceBuilder::launchRound(SchedWorkspace& w, const uint32_t* cnt, const RoundLayout& lay, uint32_t nTasks)
        {
            if (evUsed_ + 2 > w.ev.size())
                for (int i = 0; i < 2; ++i) { cudaEvent_t e; HPSDF_CUDA(cudaEventCreate(&e)); w.ev.push_back(e); }
            const hpsdf_status st = launchRoundFits(t_, o_, prog_, progSummary_, stream_, cnt, lay, nTasks, rank_, world_, w.ev[evUsed_], w.ev[evUsed_ + 1]);
            if (st != HPSDF_OK) return st;
            evUsed_ += 2;
            static const char* dbg = getenv("HPSDF_DEBUG_ROUNDS");
            if (dbg && dbg[0] == '2')
            {
                const size_t k = evUsed_ / 2 - 1;
                while (w.dbgEv.size() <= k) { cudaEvent_t e; HPSDF_CUDA(cudaEventCreate(&e)); w.dbgEv.push_back(e); }
                HPSDF_CUDA(cudaEventRecord(w.dbgEv[k], stream_));
            }
            return HPSDF_OK;
        }

        hpsdf_status DeviceBuilder::attempt(SchedWorkspace& w, uint32_t& doneCode)
        {
            SchedDev& S = w.dev;
            const hpsdf_config& cfg = t_.cfg;
            S.threshold = cfg.target_error_threshold; S.nearnessStrength = cfg.nearness_strength; S.nearnessType = cfg.nearness_type;
            S.nearnessMode = o_.nearness_mode; S.nearnessSeed = o_.nearness_seed;
            S.maxDegree = o_.max_degree; S.maxDepth = o_.max_depth; S.totalMode = o_.total_mode;
            S.minRoundJobs = o_.min_round_jobs ? o_.min_round_jobs : (progSummary_.samplesExt ? 128u : 512u);     // measured: 870 k-triangle config 9 -> 6 rounds at +0.5 % fits; 512 evaluates 60 % more
            S.speculate = o_.speculate;
            S.dealJobs = world_ > 1 ? 1u : 0u;
            S.split = S.dealJobs ? 0u : 1u;
            if (const char* dl = getenv("HPSDF_SCHED_DEAL")) S.dealJobs = dl[0] != '0' ? 1u : S.dealJobs;               // diagnostics: the multi-GPU job order on one GPU
            if (const char* sp = getenv("HPSDF_SCHED_SPLIT")) S.split = sp[0] != '0' && !S.dealJobs ? 1u : 0u;      // diagnostics: the single-CTA ingest / selection on one GPU
            if (S.dealJobs) S.split = 0u;
            S.hostHdr = w.devHdr;
            evUsed_ = 0;
            memset(&t_.stats, 0, sizeof(t_.stats));
            t_.stats.sdf_flops_per_eval = progSummary_.flopsPerEval;

            // ---- uniform start (CreateRoot + UniformlyRefine) from the templates; counters; round 0: the 4096 coarse fits at
            //      degree 2 (Octree.cpp:836-843) ------------------------------------------------------------------------------
            uint32_t cnt[kMaxDegree + 2] = { 0 };
            cnt[kCoarseDegree] = kCoarseCells;
            RoundLayout lay;
            uint64_t poolNeed = 0;
            layoutRound(cnt, 0u, lay.groupBegin, lay.groupPool, poolNeed);
            SchedCounters c0;
            memset(&c0, 0, sizeof(c0));
            c0.nNodes = kCoarseNodes; c0.nJobs = kCoarseCells; c0.poolUsed = (uint32_t)poolNeed;
            c0.roundJob0 = 0; c0.roundJobs = kCoarseCells; c0.levelKey = ~0ull; c0.levelNode = kNone;
            c0.jobsEvaluated = kCoarseCells; c0.fitsEvaluated = kCoarseCells;
            w.hostHdr->seq = 0;
            HPSDF_CUDA(launchSchedInit(S, w.tpl, c0, lay, stream_));
            t_.stats.kernel_launches++;
            HPSDF_CUDA(ws_.pool.reserve((size_t)c0.poolUsed + 1024, stream_, 0));
            HPSDF_CUDA(ws_.tasks.reserve(kCoarseCells));
            HPSDF_CUDA(ws_.recs.reserve(kCoarseCells));
            HPSDF_CUDA(launchExpandJobsDev(w.tJobs, kCoarseCells, S.layout, ws_.tasks.p, stream_));
            t_.stats.kernel_launches++;
            hpsdf_status st = launchRound(w, cnt, lay, kCoarseCells);
            if (st != HPSDF_OK) return st;

            // ---- rounds -----------------------------------------------------------------------------------------------------------
            uint32_t poolUsed = c0.poolUsed;
            uint32_t roundJobs = 0, openEstimate = kCoarseCells;
            for (uint32_t round = 0;; ++round)
            {
                S.recs = ws_.recs.p; S.pool = ws_.pool.p;
                if (S.split && round > 0) { HPSDF_CUDA(launchSchedIngest(S, roundJobs, stream_)); t_.stats.kernel_launches++; }
                HPSDF_CUDA(launchSchedRound(S, w.coarseOrder, stream_));
                t_.stats.kernel_launches++;
                if (S.split)
                {
                    // every H job of the round adds 8 entries to the open list before the selection compacts it
                    HPSDF_CUDA(launchSchedSelect(S, openEstimate + 8u * (roundJobs + 4096u), stream_));
                    t_.stats.kernel_launches += 2;
                    std::swap(S.open, S.openAlt);                 // the compacted list of the next round
                }
                if ((st = waitHeader(w, round + 1)) != HPSDF_OK) return st;
                RoundHeader h;
                memcpy(&h, (const void*)w.hostHdr, sizeof(h));
                if (getenv("HPSDF_DEBUG_ROUNDS"))
                    fprintf(stderr, "round %u: done %u, next jobs %u tasks %u, nodes %u open %u cached %u pool %u\n", round, h.done, h.nJobs, h.nTasks, h.nNodes, h.nOpen, h.nCached, h.poolUsed);
                if (h.done) { doneCode = h.done; nNodesFinal_ = h.nNodes; break; }
                roundJobs = h.nJobs; openEstimate = h.nOpen;
                if (round > 100000) { setLastError("internal: build does not converge"); return HPSDF_ERR_CUDA; }
                // next round: the layout the scheduler kernel wrote to S.layout, recomputed as a cross-check
                const uint32_t nTasks = layoutRound(h.cnt, poolUsed, lay.groupBegin, lay.groupPool, poolNeed);
                if (nTasks != h.nTasks || poolNeed != h.poolUsed) { setLastError("internal: round layout mismatch between host and device"); return HPSDF_ERR_CUDA; }
                HPSDF_CUDA(ws_.pool.reserve(poolNeed + 1024, stream_, poolUsed));
                HPSDF_CUDA(ws_.tasks.reserve(nTasks));
                HPSDF_CUDA(ws_.recs.reserve(nTasks));
                poolUsed = (uint32_t)poolNeed;
                HPSDF_CUDA(launchExpandJobsDev(S.jobsOut, h.nJobs, S.layout, ws_.tasks.p, stream_));
                t_.stats.kernel_launches++;
                t_.stats.jobs_evaluated += h.nJobs;
                if ((st = launchRound(w, h.cnt, lay, nTasks)) != HPSDF_OK) return st;
            }
            return HPSDF_OK;
        }

        // ReallocCoeffs + Query / MemoryBlock structures on the device (finish_kernels.cuh), the optional continuity solve, and
        // what comes back to the host: counters, the apply log, the near-tie log and the leaf errors (for the cut-tie log).
        hpsdf_status DeviceBuilder::finish(SchedWorkspace& w)
        {
            SchedDev& S = w.dev;
            const double tPack0 = nowMs();
            const uint32_t nN = nNodesFinal_;
            const uint32_t seq = ++w.finSeq;
            HPSDF_CUDA(launchFinishOrder(S, nN, w.sortKeys, w.sortVals, w.sortKeysAlt, w.sortValsAlt, w.leafCounter, w.sortTmp, w.sortTmpBytes,
                                         w.cstartOf, w.padOf, w.devFin, seq, stream_));
            t_.stats.kernel_launches += 6;
            // wait for the totals + counters (mapped memory), then size the tree's storage
            {
                const double t0 = nowMs();
                for (uint64_t spin = 0; w.hostFin->seq != seq; ++spin)
                    if ((spin & 0xFFF) == 0xFFF)
                    {
                        const cudaError_t q = cudaStreamQuery(stream_);
                        if (q != cudaSuccess && q != cudaErrorNotReady) return failCuda(q, "finish kernels");
                        if (nowMs() - t0 > 120000.0) { setLastError("internal: finish kernels did not answer within 120 s"); return HPSDF_ERR_CUDA; }
                    }
                std::atomic_thread_fence(std::memory_order_acquire);
            }
            const uint32_t nLeaves = w.hostFin->nLeaves;
            SchedCounters c;
            memcpy(&c, (const void*)&w.hostFin->counters, sizeof(c));
            const size_t nL = c.nLog, nD = std::min<size_t>(c.nDecision, S.capDecisions);
            t_.nNodes = nN; t_.nCoeffs = w.hostFin->nCoeffs; t_.nCoeffsPad = w.hostFin->nCoeffsPad; t_.nLogDev = nL;
            t_.nodes.clear(); t_.applyLog.clear(); t_.decisionLog.clear();
            hpsdf_status st = allocTreeBlob(t_);
            if (st != HPSDF_OK) return st;
            HPSDF_CUDA(launchEmitTree(S, nN, w.cstartOf, w.padOf, ws_.pool.p, t_.dCoeffs, t_.dNodes, t_.dNodeImage, stream_));
            t_.imageValid = true;
            t_.stats.kernel_launches++;
            // the apply log and the leaf errors stay on the device (inside the tree's allocation) until they are read
            if (nL) HPSDF_CUDA(cudaMemcpyAsync(t_.dApplyLog, S.log, nL * sizeof(hpsdf_apply_log_entry), cudaMemcpyDeviceToDevice, stream_));
            if (nL) HPSDF_CUDA(cudaMemcpyAsync(t_.dLeafErr, S.err, (size_t)nN * 8, cudaMemcpyDeviceToDevice, stream_));
            t_.logOnDevice = nL != 0;
            if (nD)
            {
                t_.decisionLog.resize(nD);
                HPSDF_CUDA(cudaMemcpyAsync(t_.decisionLog.data(), S.decisions, nD * sizeof(hpsdf_decision_log_entry), cudaMemcpyDeviceToHost, stream_));
            }
            t_.stats.pack_ms = nowMs() - tPack0;
            if (t_.cfg.continuity_enforce)
            {
                const double c0 = nowMs();
                st = continuityPostProcess(t_, o_, stream_);                                          // Octree.cpp:341-344
                if (st != HPSDF_OK) return st;
                t_.stats.continuity_ms = nowMs() - c0;
            }
            const double tFin0 = nowMs();
            HPSDF_CUDA(launchPadCoefficients(S, nN, w.cstartOf, w.padOf, t_.dCoeffs, t_.dCoeffsPad, stream_));
            HPSDF_CUDA(cudaMemcpyAsync(t_.dTop, w.tTop, 4096 * 4, cudaMemcpyDeviceToDevice, stream_));
            HPSDF_CUDA(uploadTreeView(t_, t_.dTop, stream_));
            t_.stats.kernel_launches++;
            HPSDF_CUDA(cudaStreamSynchronize(stream_));
            t_.stats.finalize_ms = nowMs() - tFin0;
            {
                static const char* dbg = getenv("HPSDF_DEBUG_ROUNDS");
                if (dbg && dbg[0] == '2' && w.dbgEv.size() >= evUsed_ / 2)
                {
                    // per round: fit launches, exchange, and the gap to the next round's launches (scheduler kernels + host turn-around)
                    cudaStreamSynchronize(stream_);
                    for (size_t k = 0; k + 1 < evUsed_; k += 2)
                    {
                        float fit = 0, comm = 0, gap = 0;
                        cudaEventElapsedTime(&fit, w.ev[k], w.ev[k + 1]);
                        cudaEventElapsedTime(&comm, w.ev[k + 1], w.dbgEv[k / 2]);
                        if (k + 2 < evUsed_) cudaEventElapsedTime(&gap, w.dbgEv[k / 2], w.ev[k + 2]);
                        fprintf(stderr, "rank %d round %zu: fits %.3f ms, exchange %.3f ms, scheduler + turn-around %.3f ms\n", rank_, k / 2, fit, comm, gap);
                    }
                }
            }
            const bool dbgRounds = getenv("HPSDF_DEBUG_ROUNDS") != nullptr;
            if (dbgRounds) printFitTimeline(rank_);
            if (dbgRounds) fprintf(stderr, "fit launches per round (ms):");
            for (size_t k = 0; k + 1 < evUsed_; k += 2)
            {
                float ms = 0.0f;
                if (cudaEventElapsedTime(&ms, w.ev[k], w.ev[k + 1]) == cudaSuccess) fitMs_ += ms;
                if (dbgRounds) fprintf(stderr, " %.3f", ms);
            }
            if (dbgRounds) fprintf(stderr, "\n");
            t_.stats.fit_kernel_ms = fitMs_;
            if (nD) std::sort(t_.decisionLog.begin(), t_.decisionLog.end(), [](const hpsdf_decision_log_entry& a, const hpsdf_decision_log_entry& b) { return a.node_idx < b.node_idx; });
            hpsdf_build_stats& s = t_.stats;
            s.jobs_evaluated += kCoarseCells;
            s.jobs_applied_p = c.appliedP; s.jobs_applied_h = c.appliedH; s.near_tie_decisions = c.nearTies;
            s.total_error = o_.total_mode == HPSDF_TOTAL_EXACT_SUM ? c.exactSum : c.total;
            s.exact_total_error = c.exactSum;
            const double thr = t_.cfg.target_error_threshold;
            const double check = o_.total_mode == HPSDF_TOTAL_EXACT_SUM ? c.exactSum : c.total;
            s.cut_margin = (thr - check) / thr;
            s.host_replay_ms = 0.0;
            // the equal-error group the cut falls into is worked out when the log is read (it needs the node array on the host)
            t_.cutLogStart = c.lastPassLogStart; t_.cutQueueEmpty = c.nOpen == 0; t_.cutLogPending = nL != 0;
            t_.cutTotalBeforeLast = c.totalBeforeLast; t_.cutCheck = check;
            s.n_nodes = nN; s.n_leaves = nLeaves; s.n_coeffs = t_.nCoeffs; ws_.lastNodeCount = nN;
            if (getenv("HPSDF_MESH_STATS")) printMeshStats();
            if (getenv("HPSDF_DEBUG_ROUNDS"))
                fprintf(stderr, "device scheduler: rounds %llu, passes %u (exact head walks %u), applied P %u H %u, retired %u, nodes %u; kernel time ingest %.1f us, passes %.1f us, select %.1f us\n",
                        (unsigned long long)s.rounds, c.passes, c.windowPasses, c.appliedP, c.appliedH, c.retired, nN, c.nsIngest * 1e-3, c.nsPasses * 1e-3, c.nsSelect * 1e-3);
            return HPSDF_OK;
        }

        hpsdf_status DeviceBuilder::run(bool& fallBack)
        {
            const double t0 = nowMs();
            fallBack = false;
            std::lock_guard<std::mutex> wsLock(*(std::mutex*)t_.ctx->wsMutex);
            stream_ = o_.stream ? (cudaStream_t)o_.stream : ws_.stream;
            if (o_.comm) { rank_ = commRank(o_.comm); world_ = commWorld(o_.comm); }
            progSummary_ = summarizeProgram(prog_);
            if (!ws_.sched) ws_.sched = new SchedWorkspace();
            SchedWorkspace& w = *(SchedWorkspace*)ws_.sched;
            hpsdf_status st = ensureTemplates(w);
            if (st != HPSDF_OK) return st;
            // the capacity only ever grows (an overflow restarts the build with four times as much and the larger arena is
            // kept), so a repeated Create never reallocates: re-sizing it from the previous node count cost C4 330 ms of
            // cudaFree + cudaMalloc in its second build
            uint32_t cap = std::max<uint32_t>(w.cap, 1u << 18);
            for (;;)
            {
                if ((st = ensureCapacity(w, cap)) != HPSDF_OK) return st;
                uint32_t done = 0;
                if ((st = attempt(w, done)) != HPSDF_OK) return st;
                if (done == 1u) break;
                if (done == 2u)
                {
                    // a list or the node arrays ran full: start over with four times the capacity
                    if (cap >= (1u << 28)) { setLastError("octree exceeds the capacity of the device scheduler"); return HPSDF_ERR_OOM; }
                    HPSDF_CUDA(cudaStreamSynchronize(stream_));
                    cap *= 4;
                    continue;
                }
                if (done == 3u) { HPSDF_CUDA(cudaStreamSynchronize(stream_)); fallBack = true; return HPSDF_OK; }   // a coarse error >= 100: the host scheduler handles it
                setLastError("internal: device scheduler stalled with nothing to evaluate");
                return HPSDF_ERR_CUDA;
            }
            if ((st = finish(w)) != HPSDF_OK) return st;
            t_.stats.total_ms = nowMs() - t0;
            return st;
        }
    }

    hpsdf_status buildOctreeDevice(hpsdf_octree& t, const hpsdf_build_opts& opts, const SdfProgramDev& prog, bool& fallBack)
    {
        DeviceBuilder b(t, opts, prog);
        return b.run(fallBack);
    }

    // Octree::Create (Octree.cpp:312-352): the device-resident scheduler unless the caller asks for the host replay
    // (hpsdf_build_opts.scheduler = 1, or strict_order = 1: sequential node numbering).
    hpsdf_status buildOctree(hpsdf_octree& t, const hpsdf_build_opts& opts, const SdfProgramDev& prog)
    {
        static const char* env = getenv("HPSDF_SCHEDULER");
        const bool host = opts.scheduler == 1u || opts.strict_order || (opts.scheduler == 0u && env && env[0] == 'h');
        if (opts.nearness_mode > HPSDF_NEARNESS_MC_COUNTER) { setLastError("unknown nearness_mode"); return HPSDF_ERR_INVALID_ARG; }
        const bool mc = opts.nearness_mode == HPSDF_NEARNESS_MC_COUNTER && t.cfg.nearness_type != HPSDF_NEARNESS_NONE;
        if (!host)
        {
            bool fallBack = false;
            const hpsdf_status st = buildOctreeDevice(t, opts, prog, fallBack);
            if (st != HPSDF_OK || !fallBack) return st;
        }
        // the host replay sees 16-byte fit records, not coefficients: it cannot sample the approximant
        if (mc) { setLastError("nearness_mode = HPSDF_NEARNESS_MC_COUNTER needs the device scheduler (scheduler = 0, strict_order = 0)"); return HPSDF_ERR_UNSUPPORTED; }
        return buildOctreeHost(t, opts, prog);
    }
}
