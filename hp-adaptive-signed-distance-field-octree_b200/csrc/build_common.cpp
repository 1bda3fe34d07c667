// build_common.cpp — round launches, ReallocCoeffs and the cut-tie log, shared by the two schedulers of Octree::Create.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include "build_common.h"
#include "comm.h"

namespace hpsdf
{
    hpsdf_status launchRoundFits(hpsdf_octree& t, const hpsdf_build_opts& o, const SdfProgramDev& prog, const ProgramSummary& ps,
                                 cudaStream_t stream, const uint32_t* cnt, const RoundLayout& lay, uint32_t nTasks, int rank, int world,
                                 cudaEvent_t evBegin, cudaEvent_t evEnd)
    {
        BuildWorkspace& ws = t.ctx->ws;
        // Sharding a round costs one grouped broadcast per (degree group, rank) and its latency. It pays when fits are
        // expensive (mesh / octree programs: 10^3-10^4 BVH queries each) or the round is large; a small round of closed-form
        // fits (tens of microseconds of kernel time) is cheaper to evaluate redundantly on every rank — identical kernels on
        // identical hardware give identical bits, so the replicas stay in lock-step without an exchange.
        const bool shard = world > 1 && (ps.samplesExt || nTasks >= (1u << 18));
        HPSDF_CUDA(cudaEventRecord(evBegin, stream));
        int groups = 0;
        for (int d = 1; d <= kMaxDegree; ++d) groups += cnt[d] != 0;
        // The launches of a round (one per degree present) are independent: they fan out over four auxiliary streams and join
        // again. Mesh / octree programs sample into a scratch buffer: their groups run concurrently when every group gets its own
        // slice of it (a mesh query is a chain of ~50-300 dependent L2 round trips, so a launch lasts at least 0.1-0.4 ms however
        // few samples it has: back to back, the groups of a small round — all of them, on 8 GPUs — just queue those latencies up).
        size_t slice[kMaxDegree + 2] = { 0 }, sliceOff[kMaxDegree + 2] = { 0 }, sliceTotal = 0;
        if (ps.samplesExt && groups > 1)
            for (int d = 1; d <= kMaxDegree; ++d)
            {
                size_t b = 0, e = cnt[d];
                if (shard) hpsdf_shard_range(cnt[d], rank, world, &b, &e);
                slice[d] = (e - b) * (size_t)fitRule(d) * fitRule(d) * fitRule(d);
                sliceOff[d] = sliceTotal;
                sliceTotal += (slice[d] + 31) & ~(size_t)31;
            }
        const bool sliced = ps.samplesExt && groups > 1 && sliceTotal <= ((size_t)1 << 28) && !getenv("HPSDF_SAMPLE_CAP");
        if (sliced) HPSDF_CUDA(reserveSampleScratch(*t.ctx, sliceTotal, stream));
        const bool fan = groups > 1 && (!ps.samplesExt || sliced);
        if (fan) HPSDF_CUDA(cudaEventRecord(ws.evFork, stream));
        int g = 0;
        bool used[4] = { false, false, false, false };
        double flops = 0.0; uint64_t evals = 0;
        for (int d = kMaxDegree; d >= 1; --d)                 // highest degree first: the longest kernels start earliest
        {
            const size_t n = cnt[d];
            if (!n) continue;
            size_t b = 0, e = n;
            if (shard) hpsdf_shard_range(n, rank, world, &b, &e);
            if (e > b)
            {
                cudaStream_t s = stream;
                if (fan)
                {
                    s = ws.aux[g & 3];
                    if (!used[g & 3]) { HPSDF_CUDA(cudaStreamWaitEvent(s, ws.evFork, 0)); used[g & 3] = true; }
                    ++g;
                }
                const hpsdf_status ls = launchFit(o.jit, d, ws.tasks.p + lay.groupBegin[d] + b, (int)(e - b), ws.pool.p, ws.recs.p, prog, t.map, *t.ctx, s,
                                                  sliced ? sliceOff[d] : 0, sliced ? slice[d] : 0, sliced ? d : 0);
                if (ls != HPSDF_OK) return ls;
                t.stats.kernel_launches++;
            }
            const double n3 = (double)fitRule(d) * fitRule(d) * fitRule(d);
            flops += (double)n * (fitFlops(d) + ps.flopsPerEval * n3);
            evals += (uint64_t)n * (uint64_t)n3;
        }
        if (fan)
            for (int i = 0; i < 4; ++i)
                if (used[i])
                {
                    HPSDF_CUDA(cudaEventRecord(ws.evJoin[i], ws.aux[i]));
                    HPSDF_CUDA(cudaStreamWaitEvent(stream, ws.evJoin[i], 0));
                }
        HPSDF_CUDA(cudaEventRecord(evEnd, stream));
        if (shard)
        {
            // every rank receives every other rank's shard: coefficients and records (replicated pool, identical replay)
            std::vector<CommSegment> segs;
            for (int d = 1; d <= kMaxDegree; ++d)
            {
                const size_t n = cnt[d];
                if (!n) continue;
                for (int r = 0; r < world; ++r)
                {
                    size_t b, e;
                    hpsdf_shard_range(n, r, world, &b, &e);
                    if (e <= b) continue;
                    segs.push_back({ ws.pool.p + lay.groupPool[d] + b * (size_t)coeffCount(d), (e - b) * (size_t)coeffCount(d), r });
                    segs.push_back({ (double*)(ws.recs.p + lay.groupBegin[d] + b), (e - b) * 2, r });
                }
            }
            const hpsdf_status cs = commBroadcastSegments(o.comm, segs, stream);
            if (cs != HPSDF_OK) return cs;
        }
        t.stats.algorithmic_flops += flops;
        t.stats.sdf_evals += evals;
        t.stats.fits_evaluated += nTasks;
        t.stats.rounds++;
        return HPSDF_OK;
    }

    hpsdf_status packCoefficients(hpsdf_octree& t, const double* pool, cudaStream_t stream)
    {
        std::vector<HostNode>& nodes = t.nodes;
        BuildWorkspace& ws = t.ctx->ws;
        std::vector<uint32_t> srcOff, dstOff, count;
        size_t cur = 0;
        std::vector<uint64_t> stack;
        for (int i = 7; i >= 0; --i) stack.push_back(nodes[0].child + (uint64_t)i);
        while (!stack.empty())
        {
            const uint64_t idx = stack.back(); stack.pop_back();
            HostNode& n = nodes[idx];
            if (n.child == kNoChild)
            {
                const uint32_t c = (uint32_t)coeffCount(n.degree);
                srcOff.push_back(n.slot); dstOff.push_back((uint32_t)cur); count.push_back(c);
                n.cstart = cur; cur += c;
            }
            else for (int i = 7; i >= 0; --i) stack.push_back(n.child + (uint64_t)i);
        }
        t.nCoeffs = cur; t.nNodes = nodes.size(); t.nCoeffsPad = paddedCoeffCount(t);
        const uint32_t nSeg = (uint32_t)srcOff.size();
        hpsdf_status st = allocTreeBlob(t);
        if (st != HPSDF_OK) return st;
        HPSDF_CUDA(ws.segs.reserve(3 * (size_t)nSeg + 16));
        HPSDF_CUDA(ws.hSegs.reserve(3 * (size_t)nSeg + 16));
        memcpy(ws.hSegs.p, srcOff.data(), nSeg * 4);
        memcpy(ws.hSegs.p + nSeg, dstOff.data(), nSeg * 4);
        memcpy(ws.hSegs.p + 2 * (size_t)nSeg, count.data(), nSeg * 4);
        HPSDF_CUDA(cudaMemcpyAsync(ws.segs.p, ws.hSegs.p, 3 * (size_t)nSeg * 4, cudaMemcpyHostToDevice, stream));
        HPSDF_CUDA(launchGatherSegments(pool, t.dCoeffs, ws.segs.p, ws.segs.p + nSeg, ws.segs.p + 2 * (size_t)nSeg, nSeg, stream));
        t.stats.kernel_launches++;
        HPSDF_CUDA(cudaStreamSynchronize(stream));       // the pinned segment staging is reused by finalizeQueryStructures
        return HPSDF_OK;
    }

    void ensureApplyLog(hpsdf_octree& t)
    {
        if (!t.logOnDevice) return;
        t.logOnDevice = false;
        t.applyLog.resize(t.nLogDev);
        cudaSetDevice(t.device);
        if (t.nLogDev && cudaMemcpy(t.applyLog.data(), t.dApplyLog, t.nLogDev * sizeof(hpsdf_apply_log_entry), cudaMemcpyDeviceToHost) != cudaSuccess)
        { cudaGetLastError(); t.applyLog.clear(); }
    }

    void ensureDecisionLog(hpsdf_octree& t)
    {
        if (!t.cutLogPending) return;
        t.cutLogPending = false;
        ensureApplyLog(t);
        if (ensureHostNodes(t) != HPSDF_OK) return;
        std::vector<double> errOf(t.nNodes);
        if (cudaMemcpy(errOf.data(), t.dLeafErr, t.nNodes * 8, cudaMemcpyDeviceToHost) != cudaSuccess) { cudaGetLastError(); return; }
        const double thr = t.cfg.target_error_threshold;
        if (t.applyLog.size() > 4096)
        {
            // the last job applied before the termination cut, with how far the total was from the threshold around it
            const hpsdf_apply_log_entry& a = t.applyLog.back();
            hpsdf_decision_log_entry e{};
            e.node_idx = a.node_idx; e.depth = t.nodes[a.node_idx].depth; e.degree = a.degree; e.chose_p = a.kind == 0; e.kind = 1;
            e.p_improvement = a.p_improvement; e.h_improvement = a.h_improvement;
            for (int k = 0; k < 3; ++k) e.centre[k] = (t.nodes[a.node_idx].mn[k] + t.nodes[a.node_idx].mx[k]) / 2.0f;
            e.relative_margin = std::min(std::fabs(t.cutTotalBeforeLast - thr), std::fabs(thr - t.cutCheck)) / thr;
            t.decisionLog.push_back(e);
        }
        logCutTieGroup(t, errOf, t.cutLogStart, t.cutQueueEmpty);
    }

    void logCutTieGroup(hpsdf_octree& t, const std::vector<double>& errOf, size_t levelLogStart, bool queueEmpty)
    {
        const std::vector<HostNode>& nodes = t.nodes;
        if (t.applyLog.empty() || queueEmpty) return;
        // the sequential loop's last pop is the smallest-error entry applied since the last sequential state
        double eLast = t.applyLog.back().initial_err;
        for (size_t k = std::min(levelLogStart, t.applyLog.size() - 1); k < t.applyLog.size(); ++k) eLast = std::min(eLast, t.applyLog[k].initial_err);
        if (!(eLast > 0.0) || std::abs(eLast - kInitialErr) < 1e-9) return;
        // errors of the members of a symmetric group agree to ~1e-10 relative (they are sums of squares of top-shell
        // coefficients that carry ~1e-16 |c000| of rounding each); the same noise separates two implementations
        const double band = 3e-9 * eLast;
        auto entry = [&](uint64_t idx, uint32_t degree, uint32_t kind, double err)
        {
            hpsdf_decision_log_entry e{};
            e.node_idx = idx; e.depth = nodes[idx].depth; e.degree = degree; e.kind = kind; e.chose_p = 0;
            for (int a = 0; a < 3; ++a) e.centre[a] = (nodes[idx].mn[a] + nodes[idx].mx[a]) / 2.0f;
            e.relative_margin = std::fabs(err - eLast) / eLast;
            t.decisionLog.push_back(e);
        };
        size_t refined = 0, unrefined = 0;
        for (size_t k = t.applyLog.size(); k-- > 0;)
        {
            const hpsdf_apply_log_entry& a = t.applyLog[k];
            if (std::fabs(a.initial_err - eLast) > band) continue;
            entry(a.node_idx, a.degree, 2u, a.initial_err);
            t.decisionLog.back().chose_p = a.kind == 0;
            ++refined;
        }
        for (uint64_t idx = 0; idx < nodes.size(); ++idx)
            if (nodes[idx].child == kNoChild && std::fabs(errOf[idx] - eLast) <= band) { entry(idx, nodes[idx].degree, 3u, errOf[idx]); ++unrefined; }
        if (unrefined == 0)
        {
            // nothing was left behind: the cut does not fall inside a tie group, drop the kind-2 entries again
            t.decisionLog.resize(t.decisionLog.size() - refined);
        }
    }
}
