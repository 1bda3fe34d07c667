// kernels.cu — the single device translation unit of libhpsdf: constant tables, all kernels, and their launchers.
// Built for sm_100a only (B200): nvcc -gencode arch=compute_100a,code=sm_100a.
#include <algorithm>
#include <vector>
#include <cuda_runtime.h>
#include "hp_common.h"
#include "device_ctx.h"

namespace hpsdf
{
    __constant__ double c_nl[kMaxDegree + 1][kMaxDepth + 1];   // NormalisedLengths (Utility.h:63-78)
    __constant__ double c_rec[kMaxDegree + 1][2];              // LegendreCoefficent (Utility.h:112-127)
}

#include "mesh_eval.cuh"
#include "query_eval.cuh"
#include "sdf_eval.cuh"
#include "mesh_sample_kernel.cuh"
#include "fit_kernels.cuh"
#include "query_kernels.cuh"
#include "continuity_kernels.cuh"
#include "points_kernel.cuh"
#include "sched_kernels.cuh"
#include "finish_kernels.cuh"
#include "mesh_build.cuh"
#include "isosurface_kernels.cuh"
#include "raycast_kernels.cuh"

namespace hpsdf
{
    void uploadConstants()
    {
        cudaMemcpyToSymbol(c_nl, tables().nl, sizeof(c_nl));
        cudaMemcpyToSymbol(c_rec, tables().rec, sizeof(c_rec));
        // LpX(a, +-1) with the reference's recurrence (Octree.cpp:988-1004); the host code is built with -ffp-contract=off
        double lp1[kMaxDegree + 1], lm1[kMaxDegree + 1];
        for (int a = 0; a <= kMaxDegree; ++a)
        {
            for (int sgn = 0; sgn < 2; ++sgn)
            {
                const double x = sgn ? -1.0 : 1.0;
                double m2 = 0.0, m1 = 1.0, l = 1.0;
                for (int i = 1; i <= a; ++i) { l = tables().rec[i][0] * x * m1 - tables().rec[i][1] * m2; m2 = m1; m1 = l; }
                (sgn ? lm1 : lp1)[a] = l;
            }
        }
        cudaMemcpyToSymbol(c_lp1, lp1, sizeof(lp1));
        cudaMemcpyToSymbol(c_lm1, lm1, sizeof(lm1));
        IsoTetCase tet[6][16];
        uint8_t chain[6][4], cellTris[256];
        isoBuildTables(tet, chain, cellTris);
        cudaMemcpyToSymbol(c_isoTet, tet, sizeof(tet));
        cudaMemcpyToSymbol(c_isoChain, chain, sizeof(chain));
        cudaMemcpyToSymbol(c_isoCellTris, cellTris, sizeof(cellTris));
        static double rayNodes[rayNodeOffset(kMaxDegree + 1)], rayBern[rayBernOffset(kMaxDegree + 1)];
        rayBuildTables(rayNodes, rayBern);
        cudaMemcpyToSymbol(c_rayNodes, rayNodes, sizeof(rayNodes));
        cudaMemcpyToSymbol(c_rayBern, rayBern, sizeof(rayBern));
    }

    // Persistent grid of 256-thread CTAs: ctasPerSm on every SM, fewer when n items fill fewer CTAs
    static unsigned persistentGrid(size_t n, int ctasPerSm, int smCount)
    {
        return (unsigned)std::min((size_t)(smCount > 0 ? smCount : 148) * ctasPerSm, (n + 255) / 256);
    }

    cudaError_t launchQuery(const DeviceTreeView& view, const double* dXyz, size_t n, double* dOut, int smCount, cudaStream_t stream)
    {
        if (!n) return cudaSuccess;
        queryKernel<<<persistentGrid(n, kQueryBlocksPerSm, smCount), kQueryThreads, 0, stream>>>(view, dXyz, n, dOut, ((uintptr_t)dXyz & 15u) == 0 ? 1 : 0);
        return cudaGetLastError();
    }

    cudaError_t launchQueryDerivatives(const DeviceTreeView& view, const double* dXyz, size_t n, double* dValue, double* dGrad,
                                       double* dHess, int smCount, cudaStream_t stream)
    {
        if (!n) return cudaSuccess;
        const int aligned = ((uintptr_t)dXyz & 15u) == 0 ? 1 : 0;
        if (dHess)
            queryDerivativesKernel<2><<<persistentGrid(n, derivBlocksPerSm(2), smCount), kQueryThreads, 0, stream>>>(view, dXyz, n, dValue,
                                                                                                                   dGrad, dHess, aligned);
        else
            queryDerivativesKernel<1><<<persistentGrid(n, derivBlocksPerSm(1), smCount), kQueryThreads, 0, stream>>>(view, dXyz, n, dValue,
                                                                                                                   dGrad, nullptr, aligned);
        return cudaGetLastError();
    }

    cudaError_t launchQueryGradient(const DeviceTreeView& view, const double* dXyz, size_t n, double* dOut, double* dGrad, cudaStream_t stream)
    {
        if (!n) return cudaSuccess;
        queryGradientKernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(view, dXyz, n, dOut, dGrad);
        return cudaGetLastError();
    }

    cudaError_t launchQueryRay(const DeviceTreeView& view, const double* dOrigins, const double* dDirs, size_t n, double tMax,
                               unsigned char* dHit, double* dT, cudaStream_t stream)
    {
        if (!n) return cudaSuccess;
        queryRayKernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(view, dOrigins, dDirs, n, tMax, dHit, dT);
        return cudaGetLastError();
    }

    cudaError_t launchRaycast(const DeviceTreeView& view, const double* dOrigins, const double* dDirs, size_t n, double tMin, double tMax,
                              double iso, double* dT, double* dNormals, int smCount, cudaStream_t stream)
    {
        if (!n) return cudaSuccess;
        raycastKernel<<<persistentGrid(n, 2, smCount), kQueryThreads, 0, stream>>>(view, dOrigins, dDirs, n, RayArgs{ tMin, tMax, iso }, dT, dNormals);
        return cudaGetLastError();
    }

    cudaError_t launchGatherSegments(const double* src, double* dst, const uint32_t* srcOff, const uint32_t* dstOff,
                                     const uint32_t* count, uint32_t nSeg, cudaStream_t stream)
    {
        if (!nSeg) return cudaSuccess;
        const unsigned blocks = (unsigned)(((size_t)nSeg * 32 + 255) / 256);
        gatherSegmentsKernel<<<blocks, 256, 0, stream>>>(src, dst, srcOff, dstOff, count, nSeg);
        return cudaGetLastError();
    }

    // COO keys are row << cooKeyShift(n) | col: as few significant bits as the matrix size allows, because every 8 of them
    // are one pass of the radix sort (n = 94 850: 34 bits = 5 passes; row << 32 | col needed 7)
    int cooKeyShift(uint32_t n)
    {
        int bits = 1;
        while (bits < 32 && (1ull << bits) < (uint64_t)n) ++bits;
        return bits;
    }

    cudaError_t launchFaceEmit(const FaceJobDev* dFaces, uint32_t nFaces, const DeviceCtx& ctx, uint64_t* keys, double* vals, uint32_t n, cudaStream_t stream)
    {
        if (!nFaces) return cudaSuccess;
        faceEmitKernel<<<nFaces, kFaceThreads, 0, stream>>>(dFaces, nFaces, ctx.fitTab.bidx, ctx.glRoots, ctx.glWeights, keys, vals, cooKeyShift(n));
        return cudaGetLastError();
    }

    cudaError_t launchDiagEmit(uint64_t* keys, double* vals, uint32_t n, double lambda, cudaStream_t stream)
    {
        if (!n) return cudaSuccess;
        diagEmitKernel<<<(n + 255) / 256, 256, 0, stream>>>(keys, vals, n, lambda, cooKeyShift(n));
        return cudaGetLastError();
    }

    cudaError_t launchScale(const double* in, double* out, uint32_t n, double s, cudaStream_t stream)
    {
        if (!n) return cudaSuccess;
        scaleKernel<<<(n + 255) / 256, 256, 0, stream>>>(in, out, n, s);
        return cudaGetLastError();
    }

    // temp-storage bytes CUB needs for the sort + reduce of nCoo entries
    size_t cooToCsrTempBytes(size_t nCoo, uint32_t n)
    {
        size_t tmpSort = 0, tmpRed = 0;
        cub::DoubleBuffer<uint64_t> kb((uint64_t*)nullptr, (uint64_t*)nullptr);
        cub::DoubleBuffer<double>   vb((double*)nullptr, (double*)nullptr);
        const int bits = cooKeyShift(n);
        cub::DeviceRadixSort::SortPairs(nullptr, tmpSort, kb, vb, (int)nCoo, 0, 2 * bits, (cudaStream_t)0);
        cub::DeviceReduce::ReduceByKey(nullptr, tmpRed, (uint64_t*)nullptr, (uint64_t*)nullptr, (double*)nullptr, (double*)nullptr,
                                       (uint32_t*)nullptr, cub::Sum(), (int)nCoo, (cudaStream_t)0);
        size_t tmpSel = 0;
        cub::DeviceSelect::Flagged(nullptr, tmpSel, (uint64_t*)nullptr, (uint8_t*)nullptr, (uint64_t*)nullptr, (uint32_t*)nullptr, (int)nCoo, (cudaStream_t)0);
        size_t m = tmpSort > tmpRed ? tmpSort : tmpRed;
        if (tmpSel > m) m = tmpSel;
        return m + 256 + nCoo;          // + one flag byte per entry
    }

    // Sort COO by (row, col), sum duplicates, build CSR. All buffers are caller-provided (the build workspace):
    // keysAlt/valsAlt/uniq: nCoo entries each; csr.val, csr.col: nCoo entries; csr.rowPtr: n + 1; dNum: one uint32.
    cudaError_t cooToCsr(uint64_t* keys, double* vals, uint64_t* keysAlt, double* valsAlt, uint64_t* uniq, uint32_t* dNum,
                         void* tmp, size_t tmpBytes, size_t nCoo, uint32_t n, CsrDev& csr, cudaStream_t stream)
    {
        cub::DoubleBuffer<uint64_t> kb(keys, keysAlt);
        cub::DoubleBuffer<double>   vb(vals, valsAlt);
        // keys are (row << bits | col) with row, col < n <= 2^bits: only the significant bits are sorted; radix sort is stable,
        // so duplicates keep their emission order and are summed in that order
        const int bits = cooKeyShift(n);
        size_t tb = tmpBytes;
        cudaError_t e = cub::DeviceRadixSort::SortPairs(tmp, tb, kb, vb, (int)nCoo, 0, 2 * bits, stream);
        tb = tmpBytes;
        if (e == cudaSuccess) e = cub::DeviceReduce::ReduceByKey(tmp, tb, kb.Current(), uniq, vb.Current(), csr.val, dNum, cub::Sum(), (int)nCoo, stream);
        uint32_t nUniq = 0;
        if (e == cudaSuccess) e = cudaMemcpyAsync(&nUniq, dNum, 4, cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        // Drop entries whose summed value is exactly 0: the dense numeric blocks carry sub-threshold entries as explicit zeros
        // (the reference never emits them, Octree.cpp:1336) and analytic low/high-face blocks cancel exactly; long rows of
        // zeros would make one thread of the row-per-thread SpMV the straggler of every CG iteration.
        uint8_t* flags = (uint8_t*)tmp + (tmpBytes - nCoo);
        uint64_t* selKeys = kb.Alternate();          // both sort buffers are free once the reduction has run
        double*   selVals = vb.Alternate();
        uint32_t nnz = 0;
        if (e == cudaSuccess && nUniq)
        {
            flagNonZeroKernel<<<(nUniq + 255) / 256, 256, 0, stream>>>(csr.val, nUniq, flags);
            e = cudaGetLastError();
            size_t tb2 = tmpBytes - nCoo;
            if (e == cudaSuccess) e = cub::DeviceSelect::Flagged(tmp, tb2, uniq, flags, selKeys, dNum, (int)nUniq, stream);
            tb2 = tmpBytes - nCoo;
            if (e == cudaSuccess) e = cub::DeviceSelect::Flagged(tmp, tb2, csr.val, flags, selVals, dNum, (int)nUniq, stream);
            if (e == cudaSuccess) e = cudaMemcpyAsync(&nnz, dNum, 4, cudaMemcpyDeviceToHost, stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
            csr.val = selVals;
        }
        if (e == cudaSuccess)
        {
            rowPtrKernel<<<(nnz + 1 + 255) / 256, 256, 0, stream>>>(selKeys, nnz, n, csr.rowPtr, csr.col, bits);
            e = cudaGetLastError();
        }
        csr.n = n; csr.nnz = nnz;
        return e;
    }

    // Face enumeration on the device (continuity_kernels.cuh): counts -> exclusive scan -> jobs. totals[0] = faces, totals[1] = COO entries
    // (without the diagonal), valid after the stream has drained; scratch: 2 * nNodes u64 + CUB temp.
    size_t faceEnumTempBytes(uint32_t nNodes)
    {
        size_t scan = 0;
        cub::DeviceScan::ExclusiveSum(nullptr, scan, (unsigned long long*)nullptr, (unsigned long long*)nullptr, (int)nNodes, (cudaStream_t)0);
        return 2 * (((size_t)nNodes * 8 + 255) & ~(size_t)255) + scan + 512;
    }

    cudaError_t launchFaceCount(const unsigned char* image, uint32_t nNodes, const uint32_t* matchCount, char* scratch, unsigned long long* hostTotals,
                                cudaStream_t stream)
    {
        const size_t arr = ((size_t)nNodes * 8 + 255) & ~(size_t)255;
        unsigned long long* counts = (unsigned long long*)scratch;
        unsigned long long* offsets = (unsigned long long*)(scratch + arr);
        void* tmp = scratch + 2 * arr;
        size_t tb = 0;
        cub::DeviceScan::ExclusiveSum(nullptr, tb, counts, offsets, (int)nNodes, stream);
        MatchTable mt{ matchCount };
        faceEnumKernel<<<(nNodes + 127) / 128, 128, 0, stream>>>(image, nNodes, mt, nullptr, 0u, counts, nullptr);
        cudaError_t e = cub::DeviceScan::ExclusiveSum(tmp, tb, counts, offsets, (int)nNodes, stream);
        if (e != cudaSuccess) return e;
        // totals = offsets[last] + counts[last]
        e = cudaMemcpyAsync(hostTotals, offsets + (nNodes - 1), 8, cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(hostTotals + 1, counts + (nNodes - 1), 8, cudaMemcpyDeviceToHost, stream);
        return e;
    }

    cudaError_t launchFaceJobs(const unsigned char* image, uint32_t nNodes, const uint32_t* matchCount, const char* scratch, uint32_t cooBase,
                               FaceJobDev* faces, cudaStream_t stream)
    {
        const size_t arr = ((size_t)nNodes * 8 + 255) & ~(size_t)255;
        const unsigned long long* offsets = (const unsigned long long*)(scratch + arr);
        MatchTable mt{ matchCount };
        faceEnumKernel<<<(nNodes + 127) / 128, 128, 0, stream>>>(image, nNodes, mt, offsets, cooBase, nullptr, faces);
        return cudaGetLastError();
    }

    int cgGridSize(uint32_t n, int smCount)
    {
        // one CTA of 1024 threads per SM (8 lanes per row), fewer if the system is small
        int grid = (int)(((size_t)n * kCgLanesPerRow + kCgThreads - 1) / kCgThreads);
        if (grid > smCount) grid = smCount;
        return grid < 1 ? 1 : grid;
    }

    // scratch: 6 n + 4 grid + 8 doubles (result[0..5], then the barrier counter); hostResult: 6 doubles (iterations, residual, ns by phase)
    cudaError_t launchCg(const CsrDev& csr, const double* b, double* x, double tol, uint32_t maxIt, int grid, double* scratch,
                         double* hostResult, cudaStream_t stream)
    {
        if (grid < 1) return cudaErrorLaunchOutOfResources;
        const size_t n = csr.n;
        CgParams P;
        P.rowPtr = csr.rowPtr; P.col = csr.col; P.val = csr.val; P.n = csr.n; P.maxIt = maxIt; P.tol = tol; P.b = b; P.x = x;
        P.r = scratch; P.p = scratch + n; P.ap = scratch + 2 * n; P.invDiag = scratch + 3 * n; P.u = scratch + 4 * n; P.s = scratch + 5 * n;
        P.partial = scratch + 6 * n; P.result = P.partial + 4 * (size_t)grid; P.barrier = (unsigned*)(P.result + 6);
        // shared-memory staging of the matrix: rows per 8-lane group, and as many entries per thread as fit (the rest is read
        // from global memory); 1.3x the mean leaves room for uneven rows
        const size_t groups = (size_t)grid * kCgThreads / kCgLanesPerRow;
        P.slots = (uint32_t)((n + groups - 1) / groups);
        const size_t smemMax = 200 * 1024;
        size_t rowBytes = (size_t)P.slots * (kCgThreads / kCgLanesPerRow) * 8;
        P.rowsStaged = rowBytes <= 96 * 1024 ? 1u : 0u;
        if (!P.rowsStaged) rowBytes = 0;
        const size_t eWant = (size_t)((double)csr.nnz / ((double)grid * kCgThreads) * 1.3) + 4;
        const size_t eFit = (smemMax - rowBytes) / ((size_t)kCgThreads * 12);
        P.eCap = (uint32_t)std::min(eWant, eFit);
        const size_t smem = (size_t)P.eCap * kCgThreads * 12 + rowBytes;
        cudaError_t e = cudaFuncSetAttribute(cgKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smemMax + 8192));
        if (e == cudaSuccess) e = cudaMemsetAsync(P.barrier, 0, 8, stream);
        void* args[] = { (void*)&P };
        if (e == cudaSuccess) e = cudaLaunchCooperativeKernel((void*)cgKernel, dim3(grid), dim3(kCgThreads), args, smem, stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(hostResult, P.result, 48, cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        return e;
    }

    // split mode (single GPU): ingest and selection as multi-block kernels around the single-CTA pass kernel
    cudaError_t launchSchedIngest(const SchedDev& S, uint32_t nJobs, cudaStream_t stream)
    {
        if (!nJobs) return cudaSuccess;
        schedIngestKernel<<<(9u * nJobs + 255u) / 256u, 256, 0, stream>>>(S);
        return cudaGetLastError();
    }
    cudaError_t launchSchedSelect(const SchedDev& S, uint32_t openEstimate, cudaStream_t stream)
    {
        uint32_t blocks = (openEstimate + kSelChunk - 1) / kSelChunk;
        blocks = blocks < 1u ? 1u : (blocks > 148u ? 148u : blocks);
        schedSelectCountKernel<<<blocks, kSchedThreads, 0, stream>>>(S);
        schedSelectScatterKernel<<<blocks, kSchedThreads, 0, stream>>>(S);
        return cudaGetLastError();
    }

    // Uniform depth-4 start of a build (CreateRoot + UniformlyRefine, Octree.cpp:792-801, 112-191) from the per-device templates,
    // the 4096 coarse jobs, the counters and the layout of round 0: one launch instead of a dozen small copies.
    __global__ void schedInitKernel(const SchedDev S, const SchedTemplates T, const SchedCounters c0, const RoundLayout lay)
    {
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i < T.nNodes)
        {
            S.cell[i] = T.cell[i]; S.child[i] = T.child[i]; S.code[i] = T.code[i]; S.depth[i] = T.depth[i]; S.degree[i] = T.degree[i]; S.state[i] = T.state[i];
            S.err[i] = 0.0;                       // internal template nodes never get one; the array is copied out whole (leaf errors of the cut-tie log)
        }
        if (i < T.nJobs)
        {
            S.jobNode[i] = T.jobNode[i]; S.jobPSlot[i] = T.jobPSlot[i]; S.jobPPos[i] = T.jobPPos[i]; S.jobFlags[i] = T.jobFlags[i];
        }
        if (i == 0) { *S.ctr = c0; *S.layout = lay; }
    }

    cudaError_t launchSchedInit(const SchedDev& S, const SchedTemplates& T, const SchedCounters& c0, const RoundLayout& lay, cudaStream_t stream)
    {
        cudaError_t e = cudaMemsetAsync(S.allCnt, 0, (char*)S.jobsOut - (char*)S.allCnt, stream);        // the three histograms are adjacent
        if (e != cudaSuccess) return e;
        schedInitKernel<<<(T.nNodes + 255) / 256, 256, 0, stream>>>(S, T, c0, lay);
        return cudaGetLastError();
    }

    cudaError_t launchSchedRound(const SchedDev& S, const uint16_t* coarseOrder, cudaStream_t stream)
    {
        static bool attrSet[16] = { false };
        int dev = 0;
        cudaGetDevice(&dev);
        if (!attrSet[dev & 15])
        {
            const cudaError_t e = cudaFuncSetAttribute(schedRoundKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSchedDynSmem);
            if (e != cudaSuccess) return e;
            attrSet[dev & 15] = true;
        }
        schedRoundKernel<<<1, kSchedThreads, kSchedDynSmem, stream>>>(S, coarseOrder);
        return cudaGetLastError();
    }

    size_t finishSortTempBytes(uint32_t capNodes)
    {
        size_t bytes = 0;
        cub::DoubleBuffer<uint32_t> kb((uint32_t*)nullptr, (uint32_t*)nullptr), vb((uint32_t*)nullptr, (uint32_t*)nullptr);
        cub::DeviceRadixSort::SortPairs(nullptr, bytes, kb, vb, (int)capNodes, 0, 31, (cudaStream_t)0);
        return bytes + 256;
    }

    // DFS order of the leaves and their coefficient offsets (finish_kernels.cuh); the totals arrive in *hdr (mapped host memory)
    cudaError_t launchFinishOrder(const SchedDev& S, uint32_t nNodes, uint32_t* keys, uint32_t* vals, uint32_t* keysAlt, uint32_t* valsAlt,
                                  uint32_t* counter, void* tmp, size_t tmpBytes, uint32_t* cstartOf, uint32_t* padOf, FinishHeader* hdr, uint32_t seq,
                                  cudaStream_t stream)
    {
        cudaError_t e = cudaMemsetAsync(counter, 0, 4, stream);
        if (e != cudaSuccess) return e;
        leafKeysKernel<<<(nNodes + 255) / 256, 256, 0, stream>>>(S.state, S.code, nNodes, keys, vals, counter);
        cub::DoubleBuffer<uint32_t> kb(keys, keysAlt), vb(vals, valsAlt);
        e = cub::DeviceRadixSort::SortPairs(tmp, tmpBytes, kb, vb, (int)nNodes, 0, 31, stream);
        if (e != cudaSuccess) return e;
        leafOffsetsKernel<<<1, 1024, 0, stream>>>(vb.Current(), counter, S.degree, cstartOf, padOf, S.ctr, hdr, seq);
        return cudaGetLastError();
    }

    cudaError_t launchEmitTree(const SchedDev& S, uint32_t nNodes, const uint32_t* cstartOf, const uint32_t* padOf, const double* pool,
                               double* packed, QNode* qnodes, unsigned char* image, cudaStream_t stream)
    {
        emitTreeKernel<<<(nNodes + 255) / 256, 256, 0, stream>>>(S, nNodes, cstartOf, padOf, pool, packed, qnodes, image);
        return cudaGetLastError();
    }

    cudaError_t launchPadCoefficients(const SchedDev& S, uint32_t nNodes, const uint32_t* cstartOf, const uint32_t* padOf, const double* packed,
                                      double* padded, cudaStream_t stream)
    {
        padCoefficientsKernel<<<(nNodes + 255) / 256, 256, 0, stream>>>(S.state, S.degree, nNodes, cstartOf, padOf, packed, padded);
        return cudaGetLastError();
    }

    // ---- hpsdf_mesh_create on the device (mesh_build.cuh) ----------------------------------------------------------------------
    size_t meshBuildTempBytes(uint32_t nTris, uint32_t nNodes)
    {
        auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
        const size_t n = nTris, n3 = 3 * (size_t)nTris;
        size_t sortEdge = 0, sortLevel = 0, scan = 0;
        cub::DoubleBuffer<unsigned long long> kb((unsigned long long*)nullptr, (unsigned long long*)nullptr);
        cub::DoubleBuffer<uint32_t> vb((uint32_t*)nullptr, (uint32_t*)nullptr);
        cub::DeviceRadixSort::SortPairs(nullptr, sortEdge, kb, vb, (int)n3, 0, 64, (cudaStream_t)0);
        cub::DeviceRadixSort::SortPairs(nullptr, sortLevel, kb, vb, (int)n, 0, 64, (cudaStream_t)0);
        cub::DeviceScan::ExclusiveSum(nullptr, scan, (uint32_t*)nullptr, (uint32_t*)nullptr, (int)nNodes, (cudaStream_t)0);
        const size_t tmp = std::max(std::max(sortEdge, sortLevel), scan);
        return al(n3 * 8) * 2 + al(n3 * 4) * 3 + al(n * 12) * 3 + al(n * 4) * 5 + al(n * 24) + al((size_t)nNodes * 4) * 7 + al(tmp) + 4096;
    }

    // Stage A: half-edges. flags (device, 2 words) must be zero; after the stream has drained, flags[0] & 1 = index out of range,
    // & 2 = an edge without a twin.
    struct MeshBuildTemp
    {
        unsigned long long *keys, *keysAlt;
        uint32_t *vals, *valsAlt, *he;
        float *tmn, *tmx, *cen;
        uint32_t *order, *orderAlt, *segBegin, *segEnd, *segNode;
        uint32_t *cbounds;
        uint32_t *parent, *nodeDepth, *arrived, *nodeBegin, *nodeEnd, *wideFlag, *wideIdx;
        void* cubTmp; size_t cubTmpBytes;
        uint32_t* flags;
    };

    MeshBuildTemp carveMeshTemp(char* arena, uint32_t nTris, uint32_t nNodes)
    {
        auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
        const size_t n = nTris, n3 = 3 * (size_t)nTris;
        MeshBuildTemp T;
        char* p = arena;
        auto take = [&](size_t bytes) { char* at = p; p += al(bytes); return at; };
        T.flags = (uint32_t*)take(256);
        T.keys = (unsigned long long*)take(n3 * 8); T.keysAlt = (unsigned long long*)take(n3 * 8);
        T.vals = (uint32_t*)take(n3 * 4); T.valsAlt = (uint32_t*)take(n3 * 4); T.he = (uint32_t*)take(n3 * 4);
        T.tmn = (float*)take(n * 12); T.tmx = (float*)take(n * 12); T.cen = (float*)take(n * 12);
        T.order = (uint32_t*)take(n * 4); T.orderAlt = (uint32_t*)take(n * 4); T.segBegin = (uint32_t*)take(n * 4); T.segEnd = (uint32_t*)take(n * 4);
        T.segNode = (uint32_t*)take(n * 4);
        T.cbounds = (uint32_t*)take(n * 24);
        T.parent = (uint32_t*)take((size_t)nNodes * 4); T.nodeDepth = (uint32_t*)take((size_t)nNodes * 4); T.arrived = (uint32_t*)take((size_t)nNodes * 4);
        T.nodeBegin = (uint32_t*)take((size_t)nNodes * 4); T.nodeEnd = (uint32_t*)take((size_t)nNodes * 4);
        T.wideFlag = (uint32_t*)take((size_t)nNodes * 4); T.wideIdx = (uint32_t*)take((size_t)nNodes * 4);
        T.cubTmp = p;
        size_t sortEdge = 0, sortLevel = 0, scan = 0;
        cub::DoubleBuffer<unsigned long long> kb((unsigned long long*)nullptr, (unsigned long long*)nullptr);
        cub::DoubleBuffer<uint32_t> vb((uint32_t*)nullptr, (uint32_t*)nullptr);
        cub::DeviceRadixSort::SortPairs(nullptr, sortEdge, kb, vb, (int)n3, 0, 64, (cudaStream_t)0);
        cub::DeviceRadixSort::SortPairs(nullptr, sortLevel, kb, vb, (int)n, 0, 64, (cudaStream_t)0);
        cub::DeviceScan::ExclusiveSum(nullptr, scan, (uint32_t*)nullptr, (uint32_t*)nullptr, (int)nNodes, (cudaStream_t)0);
        T.cubTmpBytes = std::max(std::max(sortEdge, sortLevel), scan);
        return T;
    }

    static int bitsFor(uint64_t n) { int b = 1; while (b < 63 && (1ull << b) < n) ++b; return b; }

    cudaError_t meshBuildHalfEdgesAndPseudo(const MeshBuildIn& M, const MeshBuildTemp& T, float* pseudo, cudaStream_t stream)
    {
        const uint32_t n3 = 3u * M.nTris;
        const int vb = bitsFor(M.nVerts);
        cudaError_t e = cudaMemsetAsync(T.flags, 0, 8, stream);
        if (e != cudaSuccess) return e;
        meshEdgeKeysKernel<<<(n3 + 255) / 256, 256, 0, stream>>>(M, vb, T.keys, T.vals, T.he, T.flags);
        cub::DoubleBuffer<unsigned long long> kb(T.keys, T.keysAlt);
        cub::DoubleBuffer<uint32_t> vbuf(T.vals, T.valsAlt);
        size_t tb = T.cubTmpBytes;
        e = cub::DeviceRadixSort::SortPairs(T.cubTmp, tb, kb, vbuf, (int)n3, 0, std::min(64, 2 * vb), stream);
        if (e != cudaSuccess) return e;
        meshPairKernel<<<(n3 + 255) / 256, 256, 0, stream>>>(M, vb, kb.Current(), vbuf.Current(), T.he);
        meshCheckPairedKernel<<<(n3 + 255) / 256, 256, 0, stream>>>(T.he, n3, T.flags);
        return cudaGetLastError();
    }

    // Stage B (after the flags were found clean): pseudonormals, the BVH levels, the refit. `levels` = depth of the median-split tree.
    cudaError_t meshBuildBvh(const MeshBuildIn& M, const MeshBuildTemp& T, const BvhCountTable& counts, uint32_t levels, uint32_t nNodes,
                             float* pseudo, BvhNode* nodes, const uint32_t** orderOut, cudaStream_t stream)
    {
        const uint32_t n = M.nTris;
        meshPseudoKernel<<<(n + 127) / 128, 128, 0, stream>>>(M, T.he, pseudo);
        meshTriBoundsKernel<<<(n + 255) / 256, 256, 0, stream>>>(M, T.tmn, T.tmx, T.cen, T.order, T.segBegin, T.segEnd, T.segNode);
        fillU32Kernel<<<(unsigned)(((size_t)nNodes + 255) / 256), 256, 0, stream>>>(T.nodeDepth, nNodes, 0xFFFFFFFFu);
        cudaError_t e = cudaMemsetAsync(T.arrived, 0, (size_t)nNodes * 4, stream);
        if (e != cudaSuccess) return e;
        cub::DoubleBuffer<unsigned long long> kb(T.keys, T.keysAlt);
        cub::DoubleBuffer<uint32_t> ob(T.order, T.orderAlt);
        const int endBit = 32 + bitsFor(n);
        for (uint32_t level = 0; level <= levels; ++level)
        {
            meshSegInitKernel<<<(n + 255) / 256, 256, 0, stream>>>(T.segBegin, T.segEnd, n, T.cbounds);
            meshSegBoundsKernel<<<(n + 255) / 256, 256, 0, stream>>>(ob.Current(), T.segBegin, T.segEnd, T.cen, n, T.cbounds);
            meshLevelKeysKernel<<<(n + 255) / 256, 256, 0, stream>>>(ob.Current(), T.segBegin, T.segEnd, T.segNode, T.cen, T.cbounds, n, counts, kb.Current(),
                                                                      nodes, T.parent, T.nodeDepth, level);
            if (level == levels) break;                       // the last pass only writes the leaves that appeared at the deepest level
            size_t tb = T.cubTmpBytes;
            e = cub::DeviceRadixSort::SortPairs(T.cubTmp, tb, kb, ob, (int)n, 0, std::min(64, endBit), stream);
            if (e != cudaSuccess) return e;
            meshLevelSplitKernel<<<(n + 255) / 256, 256, 0, stream>>>(T.segBegin, T.segEnd, T.segNode, n, counts);
        }
        meshRefitKernel<<<(nNodes + 255) / 256, 256, 0, stream>>>(nodes, T.parent, ob.Current(), T.tmn, T.tmx, nNodes, T.arrived);
        *orderOut = ob.Current();
        return cudaGetLastError();
    }

    // Stage C (root bounds known -> inflation margin): oriented boxes, 4-wide collapse, triangle slots.
    cudaError_t meshBuildBoxes(const MeshBuildIn& M, const MeshBuildTemp& T, const uint32_t* order, uint32_t nNodes, double inflate,
                               const BvhNode* nodes, float* obb, float* wide, float4* triVerts, cudaStream_t stream)
    {
        meshNodeRangesKernel<<<(nNodes + 255) / 256, 256, 0, stream>>>(nodes, T.parent, T.nodeDepth, nNodes, M.nTris, T.nodeBegin, T.nodeEnd, T.wideFlag);
        meshObbKernel<<<(unsigned)(((size_t)nNodes * 32 + 255) / 256), 256, 0, stream>>>(M, nodes, T.nodeBegin, T.nodeEnd, order, nNodes, inflate, obb);
        if (nNodes == 1) meshWideSingleLeafKernel<<<1, 32, 0, stream>>>(nodes, wide);
        else
        {
            size_t tb = T.cubTmpBytes;
            const cudaError_t e = cub::DeviceScan::ExclusiveSum(T.cubTmp, tb, T.wideFlag, T.wideIdx, (int)nNodes, stream);
            if (e != cudaSuccess) return e;
            meshWideKernel<<<(nNodes + 255) / 256, 256, 0, stream>>>(nodes, obb, T.wideFlag, T.wideIdx, nNodes, inflate, wide);
        }
        meshSlotsKernel<<<(M.nTris + 255) / 256, 256, 0, stream>>>(M, order, triVerts);
        return cudaGetLastError();
    }

    cudaError_t launchMeshDistance(const DeviceMeshView* dView, const float* dXyz, size_t n, float* dOut, cudaStream_t stream)
    {
        if (!n) return cudaSuccess;
        meshDistanceKernel<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(dView, dXyz, n, dOut);
        return cudaGetLastError();
    }

    // ---- hpsdf_extract_isosurface (isosurface_kernels.cuh) -------------------------------------------------------------------
    using IsoVertexCounts = thrust::transform_iterator<IsoPopc, const uint8_t*, uint32_t>;
    using IsoTriCounts = thrust::transform_iterator<IsoCellTriCount, const uint8_t*, uint32_t>;

    static size_t isoScanTempBytes(uint32_t nPoints)
    {
        size_t a = 0, b = 0;
        cub::DeviceScan::ExclusiveSum(nullptr, a, IsoVertexCounts(nullptr, IsoPopc()), (uint32_t*)nullptr, (int)nPoints, (cudaStream_t)0);
        cub::DeviceScan::ExclusiveSum(nullptr, b, IsoTriCounts(nullptr, IsoCellTriCount()), (uint32_t*)nullptr, (int)nPoints, (cudaStream_t)0);
        return std::max(a, b);
    }

    size_t isoScratchBytes(uint32_t nPoints)
    {
        auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
        const size_t n = nPoints;
        return al(n * 8) + 2 * al(n) + 2 * al(n * 4) + 256 + al(isoScanTempBytes(nPoints));
    }

    IsoScratch carveIsoScratch(void* mem, uint32_t nPoints)
    {
        auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
        const size_t n = nPoints;
        char* p = (char*)mem;
        auto take = [&](size_t bytes) { char* at = p; p += al(bytes); return at; };
        IsoScratch s;
        s.vals = (double*)take(n * 8);
        s.mask = (uint8_t*)take(n);
        s.label = (uint8_t*)take(n);
        s.vbase = (uint32_t*)take(n * 4);
        s.tbase = (uint32_t*)take(n * 4);
        s.totals = (unsigned long long*)take(256);
        s.cubTmpBytes = isoScanTempBytes(nPoints);
        s.cubTmp = take(s.cubTmpBytes);
        return s;
    }

    static uint32_t isoPoints(const IsoGrid& g) { return (g.n[0] + 1) * (g.n[1] + 1) * (g.n[2] + 1); }

    cudaError_t launchIsoGrid(const DeviceTreeView& view, const IsoGrid& g, const IsoScratch& s, int smCount, cudaStream_t stream)
    {
        isoGridKernel<<<persistentGrid(isoPoints(g), kQueryBlocksPerSm, smCount), kQueryThreads, 0, stream>>>(view, g, s.vals);
        return cudaGetLastError();
    }

    cudaError_t launchIsoCount(const IsoGrid& g, const IsoScratch& s, int smCount, unsigned long long* hostTotals, cudaStream_t stream)
    {
        const uint32_t n = isoPoints(g);
        cudaError_t e = cudaMemsetAsync(s.totals, 0, 16, stream);
        if (e != cudaSuccess) return e;
        isoCountKernel<<<persistentGrid(n, 8, smCount), 256, 0, stream>>>(g, s.vals, s.mask, s.label, s.totals);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        size_t tb = s.cubTmpBytes;
        e = cub::DeviceScan::ExclusiveSum(s.cubTmp, tb, IsoVertexCounts(s.mask, IsoPopc()), s.vbase, (int)n, stream);
        tb = s.cubTmpBytes;
        if (e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(s.cubTmp, tb, IsoTriCounts(s.label, IsoCellTriCount()), s.tbase, (int)n, stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(hostTotals, s.totals, 16, cudaMemcpyDeviceToHost, stream);
        return e;
    }

    cudaError_t launchIsoEmit(const IsoGrid& g, const IsoScratch& s, float* dVerts, uint32_t* dTris, cudaStream_t stream)
    {
        const uint32_t n = isoPoints(g), blocks = (uint32_t)(((size_t)n + 255) / 256);
        isoEmitKernel<<<blocks, 256, 0, stream>>>(g, s.vals, s.mask, s.vbase, dVerts);
        isoTriKernel<<<blocks, 256, 0, stream>>>(g, s.label, s.mask, s.vbase, s.tbase, dTris);
        return cudaGetLastError();
    }
}
