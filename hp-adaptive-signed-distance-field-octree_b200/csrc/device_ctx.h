// device_ctx.h — per-device tables and the host-callable launchers of kernels.cu.
#pragma once
#include <cuda_runtime.h>
#include <string>
#include "hp_common.h"

namespace hpsdf
{
    // One leaf-leaf shared face (ContinuityThreadPool::Input, ContinuityThreadPool.h:24-28) with everything
    // EvaluateSharedFaceIntegral{Analytically,Numerically} derives from the two nodes precomputed on the host.
    struct FaceJobDev
    {
        uint64_t cooOffset;                   // where this face's entries start in the COO arrays
        uint32_t cstartA, cstartB;            // coeffsStart of the low-side (A) and high-side (B) leaf
        uint8_t  degA, degB, depthA, depthB, dim, analytic, pad0, pad1;
        double   faceScale;                   // sharedFaceScale(t1) * sharedFaceScale(t2)   (Octree.cpp:1265-1267, 1333)
        double   invDist, invTr1, invTr2;     // 2^-depthDiff and the tangential translations (Octree.cpp:1275-1290)
    };

    template <typename T>
    struct PinnedBuf
    {
        T* p = nullptr; size_t cap = 0;
        cudaError_t reserve(size_t n)
        {
            if (n <= cap) return cudaSuccess;
            if (p) cudaFreeHost(p);
            p = nullptr;
            cap = n > cap * 2 ? n : cap * 2;
            return cudaMallocHost((void**)&p, cap * sizeof(T));
        }
    };

    template <typename T>
    struct DeviceBuf
    {
        T* p = nullptr; size_t cap = 0;
        // grows geometrically; `keep` leading elements survive a reallocation
        cudaError_t reserve(size_t n, cudaStream_t s = nullptr, size_t keep = 0)
        {
            if (n <= cap) return cudaSuccess;
            const size_t newCap = n > cap * 2 ? n : cap * 2;
            T* q = nullptr;
            cudaError_t e = cudaMalloc((void**)&q, newCap * sizeof(T));
            if (e != cudaSuccess) return e;
            if (p && keep) { e = cudaMemcpyAsync(q, p, keep * sizeof(T), cudaMemcpyDeviceToDevice, s); if (e == cudaSuccess) e = cudaStreamSynchronize(s); }
            if (p) cudaFree(p);
            p = q; cap = newCap;
            return e;
        }
    };

    // Build scratch that survives between Create calls on a device (one build at a time per device): the coefficient
    // pool, task / record buffers and their pinned host mirrors. Allocation is what dominates a millisecond-scale build.
    struct BuildWorkspace
    {
        DeviceBuf<double>    pool;
        DeviceBuf<FitTask>   tasks;
        DeviceBuf<FitRecord> recs;
        DeviceBuf<uint32_t>  segs;
        DeviceBuf<double>    samples;     // F at the Gauss-Legendre points of a chunk of fits (mesh / octree programs only)
        DeviceBuf<unsigned long long> sampleCounter;   // work counter of meshSampleKernel
        DeviceBuf<float4>    meshCut;     // per-fit cuts of the mesh BVH next to the sample scratch (mesh_sample_kernel.cuh: meshCutKernel)
        DeviceBuf<JobDesc>   jobs;
        PinnedBuf<JobDesc>   hJobs;
        PinnedBuf<FitRecord> hRecs;
        PinnedBuf<uint32_t>  hSegs;
        DeviceBuf<char>      cont;        // continuity: faces, COO, CSR, CG vectors, CUB temp
        DeviceBuf<char>      meshTmp;     // hpsdf_mesh_create: uploaded arrays + temporaries of the device mesh builder
        PinnedBuf<FaceJobDev> hFaces;
        cudaStream_t         stream = nullptr;
        cudaEvent_t          ev0 = nullptr, ev1 = nullptr;
        size_t               lastNodeCount = 0;          // nodes of the previous build (vector reservations of the next)
        void*                sched = nullptr;            // SchedWorkspace of the device-resident scheduler (build_device.cpp)
        // the fit launches of a round (one per degree) are independent: they fan out over these and join again
        cudaStream_t         aux[4] = { nullptr, nullptr, nullptr, nullptr };
        cudaEvent_t          evFork = nullptr, evJoin[4] = { nullptr, nullptr, nullptr, nullptr };
    };

    struct DeviceCtx
    {
        int           device = -1;
        FitTablesDev  fitTab{};
        void*         tabMem = nullptr;
        int           smCount = 0;
        const double* glRoots = nullptr;      // all 64 rules, rule n at n(n-1)/2, ascending nodes
        const double* glWeights = nullptr;
        BuildWorkspace ws;
        void*          wsMutex = nullptr;     // std::mutex*, serialises builds on this device
        void*          blobCache = nullptr;   // released tree allocations kept for reuse (context.cpp)
        uint32_t*      matchCount = nullptr;  // 3 x 13 x 13: entries of an analytic face block per (dim, degree, degree) (continuity.cpp)
    };

    // Tree storage comes from a small per-device cache: cudaFree + cudaMalloc per Create cost 0.3-3 ms (cudaFree synchronises
    // the device), a multiple of everything else pack does. Capacities are rounded up to 1 MiB so rebuilt trees of similar
    // size reuse the same block. Released blocks are reused by later builds on the device's build stream; callers must not
    // destroy / re-Create a tree while their own streams still run hpsdf_query_device on it (the rule of cudaFreeAsync).
    cudaError_t acquireBlob(DeviceCtx& ctx, size_t bytes, void** ptr, size_t* capacity);
    void        releaseBlob(DeviceCtx& ctx, void* ptr, size_t capacity);

    struct CsrDev
    {
        uint32_t* rowPtr = nullptr; uint32_t* col = nullptr; double* val = nullptr;
        uint32_t  n = 0, nnz = 0;
    };

    // Lazily creates the context of `device` (uploads tables and constant memory). nullptr + err on failure.
    DeviceCtx* getDeviceCtx(int device, std::string& err);

    // kernels.cu
    void        uploadConstants();
    constexpr size_t kSampleScratchDoubles = (size_t)1 << 26;      // 512 MB of samples per chunk at most
    cudaError_t launchFitKernel(int degree, const FitTask* dTasks, int n, double* pool, FitRecord* recs,
                                const SdfProgramDev& prog, bool samplesExt, const RootMap& map, DeviceCtx& ctx, cudaStream_t stream,
                                size_t sliceOffset = 0, size_t sliceDoubles = 0, int counterIdx = 0);
    cudaError_t reserveSampleScratch(DeviceCtx& ctx, size_t doubles, cudaStream_t stream);
    void        printFitTimeline(int rank);      // HPSDF_DEBUG_ROUNDS=3
    // jit.cpp: the fit launch the scheduler calls (interpreted kernels, or NVRTC-specialised ones; see hpsdf_build_opts.jit)
    hpsdf_status launchFit(uint32_t jitMode, int degree, const FitTask* dTasks, int n, double* pool, FitRecord* recs,
                           const SdfProgramDev& prog, const RootMap& map, DeviceCtx& ctx, cudaStream_t stream,
                           size_t sliceOffset = 0, size_t sliceDoubles = 0, int counterIdx = 0);
    bool        jitCompileCheck(const SdfProgramDev& prog, int degree, std::string* source, size_t* cubinBytes, std::string& why);
    void        setJitDefault(bool on);
    bool        jitDefault();
    // the fit tasks of a round's job records, at the task positions of the layout in device memory (fit_kernels.cuh)
    cudaError_t launchExpandJobsDev(const JobDesc* dJobs, uint32_t nJobs, const RoundLayout* dLayout, FitTask* dTasks, cudaStream_t stream);
    cudaError_t launchSdfEval(const SdfProgramDev& prog, const double* dXyz, size_t n, double* dOut, cudaStream_t stream);
    cudaError_t launchDfmaPeak(double* dOut, int blocks, cudaStream_t stream);
    cudaError_t launchUniformPoints(uint64_t seed, uint64_t first, size_t n, const double lo[3], const double hi[3], double* dXyz, cudaStream_t stream);
    cudaError_t launchQuery(const DeviceTreeView& view, const double* dXyz, size_t n, double* dOut, int smCount, cudaStream_t stream);
    cudaError_t launchQueryRay(const DeviceTreeView& view, const double* dOrigins, const double* dDirs, size_t n, double tMax,
                               unsigned char* dHit, double* dT, cudaStream_t stream);
    // hpsdf_raycast (raycast_kernels.cuh): first crossing of F = iso per ray; dNormals may be nullptr
    cudaError_t launchRaycast(const DeviceTreeView& view, const double* dOrigins, const double* dDirs, size_t n, double tMin, double tMax,
                              double iso, double* dT, double* dNormals, int smCount, cudaStream_t stream);
    cudaError_t launchQueryGradient(const DeviceTreeView& view, const double* dXyz, size_t n, double* dOut, double* dGrad, cudaStream_t stream);
    // hpsdf_query_derivatives (query_kernels.cuh): value, gradient, and the Hessian when dHess is not nullptr
    cudaError_t launchQueryDerivatives(const DeviceTreeView& view, const double* dXyz, size_t n, double* dValue, double* dGrad,
                                       double* dHess, int smCount, cudaStream_t stream);
    // hpsdf_extract_isosurface (isosurface_kernels.cuh): a grid of (n0+1)(n1+1)(n2+1) < 2^32 points
    struct IsoGrid
    {
        double   lo[3], h[3];     // point (i,j,k) = lo + idx * h per axis
        double   iso;
        uint32_t n[3];            // cells per axis
    };
    struct IsoScratch             // about 18 bytes per grid point
    {
        double*   vals;
        uint8_t*  mask;           // crossing owned edges, bit d-1 = direction d
        uint8_t*  label;          // inside bits of the cell whose lowest corner the point is (0 for points that are none)
        uint32_t* vbase;          // exclusive scans: first vertex / triangle of the point
        uint32_t* tbase;
        unsigned long long* totals;   // vertices, triangles (64-bit)
        void*     cubTmp;
        size_t    cubTmpBytes;
    };
    size_t      isoScratchBytes(uint32_t nPoints);
    IsoScratch  carveIsoScratch(void* mem, uint32_t nPoints);
    cudaError_t launchIsoGrid(const DeviceTreeView& view, const IsoGrid& g, const IsoScratch& s, int smCount, cudaStream_t stream);
    // masks, labels, the two scans; hostTotals[0..1] hold the vertex and triangle totals once the stream has drained
    cudaError_t launchIsoCount(const IsoGrid& g, const IsoScratch& s, int smCount, unsigned long long* hostTotals, cudaStream_t stream);
    cudaError_t launchIsoEmit(const IsoGrid& g, const IsoScratch& s, float* dVerts, uint32_t* dTris, cudaStream_t stream);
    // continuity (continuity_kernels.cuh)
    cudaError_t launchFaceEmit(const FaceJobDev* dFaces, uint32_t nFaces, const DeviceCtx& ctx, uint64_t* keys, double* vals, uint32_t n, cudaStream_t stream);
    size_t      faceEnumTempBytes(uint32_t nNodes);
    cudaError_t launchFaceCount(const unsigned char* image, uint32_t nNodes, const uint32_t* matchCount, char* scratch, unsigned long long* hostTotals,
                                cudaStream_t stream);
    cudaError_t launchFaceJobs(const unsigned char* image, uint32_t nNodes, const uint32_t* matchCount, const char* scratch, uint32_t cooBase,
                               FaceJobDev* faces, cudaStream_t stream);
    cudaError_t launchDiagEmit(uint64_t* keys, double* vals, uint32_t n, double lambda, cudaStream_t stream);
    size_t      cooToCsrTempBytes(size_t nCoo, uint32_t n);
    // sort COO by (row, col), sum duplicates, build CSR; every buffer comes from the caller (build workspace)
    cudaError_t cooToCsr(uint64_t* keys, double* vals, uint64_t* keysAlt, double* valsAlt, uint64_t* uniq, uint32_t* dNum,
                         void* tmp, size_t tmpBytes, size_t nCoo, uint32_t n, CsrDev& csr, cudaStream_t stream);
    int         cgGridSize(uint32_t n, int smCount);
    // (A) x = b by preconditioned CG from the guess in x; scratch: 4 n + 3 grid + 2 doubles;
    // hostResult[0] = iterations, [1] = relative residual
    cudaError_t launchCg(const CsrDev& csr, const double* b, double* x, double tol, uint32_t maxIt, int grid, double* scratch,
                         double* hostResult, cudaStream_t stream);
    cudaError_t launchScale(const double* in, double* out, uint32_t n, double s, cudaStream_t stream);
    // dst[dstOff[s] + i] = src[srcOff[s] + i], i < count[s], for nSeg segments (ReallocCoeffs, Octree.cpp:474-555, on device)
    cudaError_t launchGatherSegments(const double* src, double* dst, const uint32_t* srcOff, const uint32_t* dstOff,
                                     const uint32_t* count, uint32_t nSeg, cudaStream_t stream);
}
