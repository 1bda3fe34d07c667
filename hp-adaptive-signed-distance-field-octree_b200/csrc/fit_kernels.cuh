// fit_kernels.cuh — host launchers of fitKernel<D, EXT> (the kernel itself: fit_kernel_body.cuh).
#pragma once
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cuda_runtime.h>
#include "hp_common.h"
#include "device_ctx.h"
#include "fit_kernel_body.cuh"

namespace hpsdf
{
    // ---- mesh / octree programs: F is sampled by a separate kernel -------------------------------------------------------
    // A BVH closest-triangle query (mesh_eval.cuh) or a tree Query is latency-bound pointer chasing that wants every warp
    // slot of the SM; inside the fit kernel (one CTA per fit, a thread per (i, j) column walking k, 168 registers with the
    // evaluators inlined) it ran at 12 warps per SM and 2.6e7 mesh samples/s. So for these programs the round is two
    // launches per chunk: sampleKernel, one thread per Gauss-Legendre sample at full occupancy, writes F to a scratch
    // buffer laid out [fit][k][j][i]; fitKernel<D, true> reads it back coalesced (16 bytes of HBM traffic per sample —
    // nothing next to a traversal). Closed-form programs keep sampling in registers inside the fit kernel.
    __global__ void __launch_bounds__(256) sampleKernel(const FitTask* __restrict__ tasks, unsigned long long nSamples, int D,
                                                        const SdfProgramDev prog, const RootMap map, const FitTablesDev tab,
                                                        double* __restrict__ samples)
    {
        __shared__ SdfProgramSmem sProg;
        stageProgram(sProg, prog);
        __syncthreads();
        const unsigned n = (unsigned)fitRule(D), n2 = n * n, n3 = n2 * n;
        const double* __restrict__ roots = tab.roots[D];
        // warp-uniform trip count (lanes past the end redo the last sample), so the traversals of a warp stay in step
        for (unsigned long long base = (unsigned long long)blockIdx.x * blockDim.x; base < nSamples; base += (unsigned long long)gridDim.x * blockDim.x)
        {
            const unsigned long long gi = base + threadIdx.x;
            const bool valid = gi < nSamples;
            const unsigned long long g = valid ? gi : nSamples - 1;
            const unsigned fit = (unsigned)(g / n3), s = (unsigned)(g - (unsigned long long)fit * n3);
            const unsigned k = s / n2, col = s - k * n2, j = col / n, i = col - j * n;
            const float4 cell = *reinterpret_cast<const float4*>(&tasks[fit]);          // cx, cy, cz, half
            const double half = (double)cell.w;
            const double X = samplePos(roots[i], half, (double)cell.x, map.sizes[0], map.centre[0]);
            const double Y = samplePos(roots[j], half, (double)cell.y, map.sizes[1], map.centre[1]);
            const double Z = samplePos(roots[k], half, (double)cell.z, map.sizes[2], map.centre[2]);
            const double f = sdfEval<1>(sProg, X, Y, Z);
            if (valid) samples[g] = f;
        }
    }

    // HPSDF_MESH_STATS=1: a 64-word device buffer collecting the node-step histogram of meshSampleKernel (words 0-41) and
    // its event counts (words 42.., mesh_sample_kernel.cuh: MeshStat), printed by hpsdf_debug_mesh_stats; nullptr otherwise.
    static unsigned long long* g_meshStats[16] = { nullptr };
    static unsigned long long* meshStatsBuffer()
    {
        static const bool on = getenv("HPSDF_MESH_STATS") != nullptr;
        if (!on) return nullptr;
        int dev = 0;
        cudaGetDevice(&dev);
        if (!g_meshStats[dev & 15])
        {
            if (cudaMalloc((void**)&g_meshStats[dev & 15], 64 * 8) != cudaSuccess) return nullptr;
            cudaMemset(g_meshStats[dev & 15], 0, 64 * 8);
        }
        return g_meshStats[dev & 15];
    }
    void printMeshStats()
    {
        int dev = 0;
        cudaGetDevice(&dev);
        if (!g_meshStats[dev & 15]) return;
        unsigned long long h[64];
        cudaMemcpy(h, g_meshStats[dev & 15], sizeof(h), cudaMemcpyDeviceToHost);
        cudaMemset(g_meshStats[dev & 15], 0, 64 * 8);
        unsigned long long n = 0;
        for (int b = 0; b < 40; ++b) n += h[b];
        fprintf(stderr, "meshSampleKernel: %llu queries, mean %.1f node steps, max %llu; queries by steps:", n, n ? (double)h[40] / n : 0.0, h[41]);
        for (int b = 0; b < 40; ++b) if (h[b]) fprintf(stderr, " <%llu: %llu", 1ull << b, h[b]);
        fprintf(stderr, "\n");
        // the event counts include the work of tail-phase helpers, which the histogram above leaves out
        const unsigned long long* c = h + kMeshStatWord;
        const double q = n ? (double)n : 1.0;
        fprintf(stderr, "meshSampleKernel per query: %.2f node steps = %.2f node visits + %.2f stale pops (%.2f more entries dropped with them); "
                        "%.2f leaves tested, %.2f dequeued already pruned; %.1f lanes per node iteration, %.1f per triangle iteration\n",
                (c[kStatNodeVisit] + c[kStatStalePop]) / q, c[kStatNodeVisit] / q, c[kStatStalePop] / q, c[kStatGroupDrop] / q,
                c[kStatLeafTest] / q, c[kStatLeafPruned] / q,
                c[kStatWarpNodeIter] ? (double)(c[kStatNodeVisit] + c[kStatStalePop]) / c[kStatWarpNodeIter] : 0.0,
                c[kStatWarpTriIter] ? (double)(c[kStatLeafTest] + c[kStatLeafPruned]) / c[kStatWarpTriIter] : 0.0);
        const unsigned long long* k = h + kCutStatWord;
        if (k[3])
            fprintf(stderr, "meshCutKernel: %llu fits, mean %.2f cut entries, max %llu; %.1f %% of the cuts are still the root's children\n",
                    k[3], (double)k[0] / k[3], k[1], 100.0 * k[2] / k[3]);
    }

    // HPSDF_DEBUG_ROUNDS=3: events around the sample and fit kernels of every degree group (diagnostics only)
    struct FitTimelineEntry { cudaEvent_t a, b, c; int degree; unsigned long long samples; size_t fits; };
    static std::vector<FitTimelineEntry> g_fitTimeline;
    static bool fitTimelineOn()
    {
        static const char* dbg = getenv("HPSDF_DEBUG_ROUNDS");
        return dbg && dbg[0] == '3';
    }
    void printFitTimeline(int rank)
    {
        if (!fitTimelineOn()) return;
        cudaDeviceSynchronize();
        for (size_t i = 0; i < g_fitTimeline.size(); ++i)
        {
            FitTimelineEntry& e = g_fitTimeline[i];
            float s = 0, f = 0, fromFirst = 0;
            cudaEventElapsedTime(&s, e.a, e.b); cudaEventElapsedTime(&f, e.b, e.c);
            cudaEventElapsedTime(&fromFirst, g_fitTimeline[0].a, e.a);
            fprintf(stderr, "rank %d t=%8.3f ms: degree %d, %zu fits, %llu samples: sample kernel %.3f ms, fit kernel %.3f ms\n", rank, fromFirst, e.degree, e.fits, e.samples, s, f);
            cudaEventDestroy(e.a); cudaEventDestroy(e.b); cudaEventDestroy(e.c);
        }
        g_fitTimeline.clear();
    }

    template <int D, bool EXT>
    static cudaError_t launchOne(const FitTask* dTasks, int n, double* pool, FitRecord* recs, const SdfProgramDev& prog,
                                 const RootMap& map, const FitTablesDev& tab, double* samples, size_t sampleCap, float4* cut,
                                 unsigned long long* counter, int smCount, cudaStream_t stream)
    {
        constexpr size_t smem = fitSmemDoubles(D) * sizeof(double);
        static bool attrSet[16] = { false };
        int dev = 0;
        cudaGetDevice(&dev);
        if (!attrSet[dev & 15])
        {
            cudaError_t e = cudaFuncSetAttribute(fitKernel<D, EXT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            attrSet[dev & 15] = true;
        }
        if constexpr (!EXT)
        {
            fitKernel<D, false><<<(n + fitGroup(D) - 1) / fitGroup(D), fitThreads(D), smem, stream>>>(dTasks, pool, recs, prog, map, tab, nullptr, n);
            return cudaGetLastError();
        }
        else
        {
            constexpr size_t n3 = (size_t)fitRule(D) * fitRule(D) * fitRule(D);
            // the cut records of a chunk are indexed in bits 0-27 of a stack entry (mesh_sample_kernel.cuh)
            const size_t chunk = std::min(sampleCap / n3, ((size_t)1 << 28) / kCutStride - 1);
            if (!samples || !cut || !chunk) return cudaErrorInvalidValue;
            for (size_t b = 0; b < (size_t)n; b += chunk)
            {
                const size_t m = std::min(chunk, (size_t)n - b);
                const unsigned long long total = (unsigned long long)m * n3;
                const unsigned long long sms = (unsigned long long)(smCount > 0 ? smCount : 148);
                FitTimelineEntry tl{};
                if (fitTimelineOn())
                {
                    cudaEventCreate(&tl.a); cudaEventCreate(&tl.b); cudaEventCreate(&tl.c);
                    tl.degree = D; tl.samples = total; tl.fits = m;
                    cudaEventRecord(tl.a, stream);
                }
                if (prog.n == 1 && prog.instr[0].op == HPSDF_PRIM_MESH)
                {
                    // the whole program is one mesh: the warp-scheduled traversal kernel (mesh_sample_kernel.cuh)
                    const unsigned grab = 32u;      // one query per lane per grab: a larger grab leaves a tail of sequential ~1 ms queries at the end of the launch
                    const unsigned long long want = (total + 8ull * grab - 1) / (8ull * grab);
                    cudaError_t e = cudaMemsetAsync(counter, 0, sizeof(unsigned long long), stream);
                    if (e != cudaSuccess) return e;
                    // 4 CTAs of 256 per SM (64 registers) and "test triangles once 12 lanes have one waiting" measured best on
                    // B200 (870 k-triangle mesh, binary tree: 2 CTAs/24 lanes 113 ms, 3/24 101 ms, 4/24 95 ms, 4/12 88 ms, 4/4 95 ms;
                    // 4-wide tree: 8 or 12 lanes 62.8 ms, 16 63.9, 20 66.3, 24 70.5). With leaves queued straight from the node step
                    // into an 8-entry queue, 16 lanes measured best on C3: 8 / 12 / 16 / 20 lanes 54.7 / 50.7 / 49.1 / 49.2 ms.
                    constexpr int triThreshold = 16;
                    unsigned long long* stats = meshStatsBuffer();
                    const size_t statSmem = stats ? (size_t)kMeshStatCount * 256 * sizeof(unsigned) : 0;
                    const DeviceMeshView* mesh = (const DeviceMeshView*)prog.instr[0].handle;
                    // every sample of a fit starts from the fit's cut of the tree (HPSDF_MESH_NO_CUT: from the root, for A/B runs)
                    const bool useCut = getenv("HPSDF_MESH_NO_CUT") == nullptr;
                    if (useCut) meshCutKernel<<<(unsigned)((m + 3) / 4), 128, 0, stream>>>(dTasks + b, (unsigned)m, D, mesh, map, tab, cut, stats);
                    meshSampleKernel<<<(unsigned)std::min(want, sms * 4), 256, statSmem, stream>>>(dTasks + b, total, D, mesh, map, tab, samples, counter, grab, triThreshold,
                                                                                                 getenv("HPSDF_MESH_NO_HANDOVER") ? 0 : 1, useCut ? cut : nullptr, stats);
                }
                else
                {
                    const unsigned long long want = (total + 255) / 256;
                    sampleKernel<<<(unsigned)std::min(want, sms * 64), 256, 0, stream>>>(dTasks + b, total, D, prog, map, tab, samples);
                }
                if (tl.a) cudaEventRecord(tl.b, stream);
                fitKernel<D, true><<<(unsigned)((m + fitGroup(D) - 1) / fitGroup(D)), fitThreads(D), smem, stream>>>(dTasks + b, pool, recs, prog, map, tab, samples, (int)m);
                if (tl.a) { cudaEventRecord(tl.c, stream); g_fitTimeline.push_back(tl); }
            }
            return cudaGetLastError();
        }
    }

    template <bool EXT>
    static cudaError_t launchFitKernelT(int degree, const FitTask* dTasks, int n, double* pool, FitRecord* recs, const SdfProgramDev& prog,
                                        const RootMap& map, const FitTablesDev& tab, double* samples, size_t sampleCap, float4* cut,
                                        unsigned long long* counter, int smCount, cudaStream_t stream)
    {
        if (n <= 0) return cudaSuccess;
        switch (degree)
        {
#define HPSDF_FIT_CASE(d) case d: return launchOne<d, EXT>(dTasks, n, pool, recs, prog, map, tab, samples, sampleCap, cut, counter, smCount, stream);
            HPSDF_FIT_CASE(1) HPSDF_FIT_CASE(2) HPSDF_FIT_CASE(3) HPSDF_FIT_CASE(4) HPSDF_FIT_CASE(5) HPSDF_FIT_CASE(6)
            HPSDF_FIT_CASE(7) HPSDF_FIT_CASE(8) HPSDF_FIT_CASE(9) HPSDF_FIT_CASE(10) HPSDF_FIT_CASE(11)
#undef HPSDF_FIT_CASE
            default: return cudaErrorInvalidValue;
        }
    }

    // cut records (meshCutKernel) that go with `doubles` of sample scratch: a slice at sample offset o owns the records from
    // cutOffset(o) on, and no chunk of it has more fits than the slice has multiples of the smallest fit's sample count
    static size_t cutFloat4s(size_t doubles) { return (doubles / kCutSamplesPerFit + 1) * kCutStride * 8; }
    static size_t cutOffset(size_t sampleOffset) { return sampleOffset / kCutSamplesPerFit * kCutStride * 8; }

    // Sample scratch of mesh / octree programs and the cut records next to it: grow-only, sized by the caller BEFORE a round
    // whose degree groups run concurrently (a reallocation inside the round would pull the buffers from under the launches in
    // flight).
    cudaError_t reserveSampleScratch(DeviceCtx& ctx, size_t doubles, cudaStream_t stream)
    {
        if (ctx.ws.samples.cap < doubles || ctx.ws.meshCut.cap < cutFloat4s(doubles))
        {
            cudaError_t e = cudaStreamSynchronize(stream);
            if (e == cudaSuccess) e = ctx.ws.samples.reserve(doubles);
            if (e == cudaSuccess) e = ctx.ws.meshCut.reserve(cutFloat4s(doubles));
            if (e != cudaSuccess) return e;
        }
        if (!ctx.ws.sampleCounter.p) return ctx.ws.sampleCounter.reserve(32);
        return cudaSuccess;
    }

    // Launch the fits of one degree. dTasks: n tasks, all with task.degree == degree. Programs with mesh / octree
    // primitives need the device context's sample scratch: the whole buffer in chunks (sliceDoubles == 0), or — when the
    // degree groups of a round run on different streams — the caller's slice [sliceOffset, sliceOffset + sliceDoubles) of a
    // buffer it reserved with reserveSampleScratch, and its own work counter. samplesExt: summarizeProgram(prog).samplesExt.
    cudaError_t launchFitKernel(int degree, const FitTask* dTasks, int n, double* pool, FitRecord* recs,
                                const SdfProgramDev& prog, bool samplesExt, const RootMap& map, DeviceCtx& ctx, cudaStream_t stream,
                                size_t sliceOffset, size_t sliceDoubles, int counterIdx)
    {
        if (!samplesExt) return launchFitKernelT<false>(degree, dTasks, n, pool, recs, prog, map, ctx.fitTab, nullptr, 0, nullptr, nullptr, ctx.smCount, stream);
        const size_t n3 = (size_t)fitRule(degree) * fitRule(degree) * fitRule(degree);
        if (sliceDoubles)
        {
            if (sliceDoubles < (size_t)std::max(n, 1) * n3 || sliceOffset + sliceDoubles > ctx.ws.samples.cap || !ctx.ws.sampleCounter.p) return cudaErrorInvalidValue;
            return launchFitKernelT<true>(degree, dTasks, n, pool, recs, prog, map, ctx.fitTab, ctx.ws.samples.p + sliceOffset, sliceDoubles,
                                          ctx.ws.meshCut.p + cutOffset(sliceOffset), ctx.ws.sampleCounter.p + counterIdx, ctx.smCount, stream);
        }
        // chunk size limit; HPSDF_SAMPLE_CAP (doubles, read per call) lets the tests force the multi-chunk path on small inputs
        size_t limit = kSampleScratchDoubles;
        if (const char* env = getenv("HPSDF_SAMPLE_CAP")) limit = (size_t)strtoull(env, nullptr, 10);
        limit = std::max(limit, n3);
        const size_t want = std::min<size_t>((size_t)std::max(n, 1) * n3, limit);
        const cudaError_t e = reserveSampleScratch(ctx, want, stream);
        if (e != cudaSuccess) return e;
        return launchFitKernelT<true>(degree, dTasks, n, pool, recs, prog, map, ctx.fitTab, ctx.ws.samples.p, std::min(ctx.ws.samples.cap, limit),
                                      ctx.ws.meshCut.p, ctx.ws.sampleCounter.p, ctx.smCount, stream);
    }

    // ---- job records -> fit tasks ------------------------------------------------------------------------------------
    // A scheduler writes one 32-byte JobDesc per refinement job and the round's layout; the 9 task descriptors of a job are
    // derived here (cells are dyadic: child centre = c +- h/2, exact in f32 — the values CornerAABB + center() give,
    // Octree.cpp:1096-1112).
    __global__ void expandJobsDevKernel(const JobDesc* __restrict__ jobs, uint32_t nJobs, const RoundLayout* __restrict__ lay, FitTask* __restrict__ tasks)
    {
        const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
        const uint32_t ji = t / 9u, c = t - ji * 9u;
        if (ji >= nJobs) return;
        const JobDesc j = jobs[ji];
        FitTask o;
        int d;
        uint32_t pos;
        if (c < 8u)
        {
            if (!(j.flags & 1u)) return;
            const float q = j.half * 0.5f;
            d = j.degree; pos = j.hPos + c;
            o.cx = j.cx + ((c & 1u) ? q : -q); o.cy = j.cy + ((c & 2u) ? q : -q); o.cz = j.cz + ((c & 4u) ? q : -q); o.half = q;
            o.src = kNoSrc; o.depth = (uint8_t)(j.depth + 1); o.degreeIn = 0;
        }
        else
        {
            if (!(j.flags & 6u)) return;
            const bool coarse = (j.flags & 4u) != 0;
            d = coarse ? kCoarseDegree : j.degree + 1; pos = j.pPos;
            o.cx = j.cx; o.cy = j.cy; o.cz = j.cz; o.half = j.half;
            o.src = coarse ? kNoSrc : j.src; o.depth = j.depth; o.degreeIn = coarse ? 0 : j.degree;
        }
        o.out = lay->groupPool[d] + (pos - lay->groupBegin[d]) * (uint32_t)coeffCount(d);
        o.degree = (uint8_t)d; o.pad = 0; o.rec = pos;
        tasks[pos] = o;
    }

    cudaError_t launchExpandJobsDev(const JobDesc* dJobs, uint32_t nJobs, const RoundLayout* dLayout, FitTask* dTasks, cudaStream_t stream)
    {
        if (!nJobs) return cudaSuccess;
        expandJobsDevKernel<<<(nJobs * 9u + 255u) / 256u, 256, 0, stream>>>(dJobs, nJobs, dLayout, dTasks);
        return cudaGetLastError();
    }

    // ---- program evaluation at arbitrary points (hpsdf_sdf_eval) and the FP64 peak probe ---------------------------
    __global__ void sdfEvalKernel(const SdfProgramDev prog, const double* __restrict__ xyz, size_t n, double* __restrict__ out)
    {
        __shared__ SdfProgramSmem sProg;
        stageProgram(sProg, prog);
        __syncthreads();
        const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i < n) out[i] = sdfEval<1>(sProg, xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]);
    }

    cudaError_t launchSdfEval(const SdfProgramDev& prog, const double* dXyz, size_t n, double* dOut, cudaStream_t stream)
    {
        if (!n) return cudaSuccess;
        sdfEvalKernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(prog, dXyz, n, dOut);
        return cudaGetLastError();
    }

    // 8 independent DFMA chains per thread, 4096 iterations: 2 * 8 * 4096 flops per thread.
    __global__ void __launch_bounds__(256) dfmaPeakKernel(double* out, double a, double b)
    {
        double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
        #pragma unroll 1
        for (int i = 0; i < 512; ++i)
        {
            #pragma unroll
            for (int u = 0; u < 8; ++u)
            {
                x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
                x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
            }
        }
        out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    }

    cudaError_t launchDfmaPeak(double* dOut, int blocks, cudaStream_t stream)
    {
        dfmaPeakKernel<<<blocks, 256, 0, stream>>>(dOut, 0.999999, 1e-9);
        return cudaGetLastError();
    }
}
