// capi.cpp — the extern "C" surface declared in include/hpsdf.h.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>
#include "octree.h"

namespace hpsdf { void printMeshStats(); }      // fit_kernels.cuh (HPSDF_MESH_STATS)
using namespace hpsdf;

namespace
{
    hpsdf_status needDevice(int device, DeviceCtx** ctx)
    {
        std::string err;
        DeviceCtx* c = getDeviceCtx(device, err);
        if (!c) { setLastError(err); return HPSDF_ERR_NO_DEVICE; }
        *ctx = c;
        return HPSDF_OK;
    }

    hpsdf_build_opts normalisedOpts(const hpsdf_build_opts* in)
    {
        hpsdf_build_opts o;
        hpsdf_build_opts_default(&o);
        if (in) memcpy(&o, in, std::min<size_t>(in->struct_size ? in->struct_size : sizeof(o), sizeof(o)));
        o.struct_size = sizeof(o);
        if (o.max_degree == 0 || o.max_degree > (uint32_t)kMaxDegree - 1) o.max_degree = kMaxDegree - 1;
        if (o.max_degree < (uint32_t)kCoarseDegree) o.max_degree = kCoarseDegree;
        if (o.max_depth == 0 || o.max_depth > (uint32_t)kMaxDepth) o.max_depth = kMaxDepth;
        if (o.max_depth < (uint32_t)kCoarseDepth) o.max_depth = kCoarseDepth;
        return o;
    }
}

extern "C"
{
    HPSDF_API const char* hpsdf_status_string(hpsdf_status s)
    {
        switch (s)
        {
            case HPSDF_OK:              return "ok";
            case HPSDF_ERR_INVALID_ARG: return "invalid argument";
            case HPSDF_ERR_NO_DEVICE:   return "no CUDA device (there is no CPU path)";
            case HPSDF_ERR_CUDA:        return "CUDA error";
            case HPSDF_ERR_BAD_BLOCK:   return "MemoryBlock does not parse";
            case HPSDF_ERR_UNSUPPORTED: return "unsupported";
            case HPSDF_ERR_COMM:        return "communicator error";
            case HPSDF_ERR_OOM:         return "out of memory";
            case HPSDF_ERR_MESH:        return "mesh is not a closed manifold";
        }
        return "unknown status";
    }

    HPSDF_API const char* hpsdf_last_error(void) { return lastError().c_str(); }
    HPSDF_API const char* hpsdf_version(void) { return "hpsdf-b200 0.1 (sm_100a)"; }

    HPSDF_API int hpsdf_device_count(void)
    {
        int n = 0;
        if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
        return n;
    }

    // Config::Config() (Config.cpp:5-14)
    HPSDF_API void hpsdf_config_default(hpsdf_config* cfg)
    {
        if (!cfg) return;
        memset(cfg, 0, sizeof(*cfg));
        cfg->target_error_threshold = std::pow(10, -10);
        cfg->nearness_type          = HPSDF_NEARNESS_NONE;
        cfg->continuity_enforce     = 1;
        cfg->continuity_strength    = 8.0;
        const unsigned hc = std::thread::hardware_concurrency();
        cfg->thread_count           = hc != 0 ? hc : 1;
        for (int i = 0; i < 3; ++i) { cfg->root_min[i] = -0.5f; cfg->root_max[i] = 0.5f; }
        cfg->enable_logging         = 0;
    }

    // Config::IsValid() (Config.cpp:17-32)
    HPSDF_API hpsdf_status hpsdf_config_validate(const hpsdf_config* cfg)
    {
        if (!cfg) { setLastError("config is null"); return HPSDF_ERR_INVALID_ARG; }
        const char* why = nullptr;
        const float vol = (cfg->root_max[0] - cfg->root_min[0]) * ((cfg->root_max[1] - cfg->root_min[1]) * (cfg->root_max[2] - cfg->root_min[2]));
        if (!(cfg->target_error_threshold > 0.0)) why = "targetErrorThreshold must be > 0";
        else if (!(cfg->thread_count > 0)) why = "threadCount must be > 0";
        else if (!(vol > 0.0f)) why = "root volume must be > 0";
        else if (cfg->nearness_type > HPSDF_NEARNESS_EXPONENTIAL) why = "unknown nearnessWeighting.type";
        else if (cfg->nearness_type != HPSDF_NEARNESS_NONE && !(cfg->nearness_strength > 0.0)) why = "nearnessWeighting.strength must be > 0";
        else if (cfg->continuity_enforce && !(cfg->continuity_strength > 0.0)) why = "continuity.strength must be > 0";
        if (why) { setLastError(why); return HPSDF_ERR_INVALID_ARG; }
        return HPSDF_OK;
    }

    HPSDF_API void hpsdf_build_opts_default(hpsdf_build_opts* o)
    {
        if (!o) return;
        memset(o, 0, sizeof(*o));
        o->struct_size   = sizeof(*o);
        o->max_degree    = kMaxDegree - 1;      // Octree.cpp:600
        o->max_depth     = kMaxDepth;
        o->nearness_mode = HPSDF_NEARNESS_EXACT_MEAN;
        o->total_mode    = HPSDF_TOTAL_REFERENCE;
        o->cg_tolerance  = 0.0;
        o->device        = -1;
    }

    HPSDF_API hpsdf_status hpsdf_sdf_eval(const hpsdf_sdf_program* prog, const double* xyz, size_t n, double* out, int device)
    {
        if (!xyz || !out) { setLastError("null pointer"); return HPSDF_ERR_INVALID_ARG; }
        DeviceCtx* ctx = nullptr;
        hpsdf_status st = needDevice(device, &ctx);
        if (st != HPSDF_OK) return st;
        SdfProgramDev dp;
        if ((st = resolveProgram(prog, ctx->device, dp)) != HPSDF_OK) return st;
        if (!n) return HPSDF_OK;
        double *dIn = nullptr, *dOut = nullptr;
        HPSDF_CUDA(cudaMalloc((void**)&dIn, n * 24));
        cudaError_t e = cudaMalloc((void**)&dOut, n * 8);
        if (e == cudaSuccess) e = cudaMemcpy(dIn, xyz, n * 24, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = launchSdfEval(dp, dIn, n, dOut, nullptr);
        if (e == cudaSuccess) e = cudaMemcpy(out, dOut, n * 8, cudaMemcpyDeviceToHost);
        cudaFree(dIn); cudaFree(dOut);
        if (e != cudaSuccess) return failCuda(e, "hpsdf_sdf_eval");
        return HPSDF_OK;
    }

    HPSDF_API hpsdf_status hpsdf_create(const hpsdf_config* cfg, const hpsdf_build_opts* opts, const hpsdf_sdf_program* prog, hpsdf_octree** out)
    {
        if (!out) { setLastError("out is null"); return HPSDF_ERR_INVALID_ARG; }
        *out = nullptr;
        hpsdf_status st = hpsdf_config_validate(cfg);
        if (st != HPSDF_OK) return st;
        const hpsdf_build_opts o = normalisedOpts(opts);
        DeviceCtx* ctx = nullptr;
        if ((st = needDevice(o.device, &ctx)) != HPSDF_OK) return st;
        SdfProgramDev dp;
        if ((st = resolveProgram(prog, ctx->device, dp)) != HPSDF_OK) return st;
        hpsdf_octree* t = new hpsdf_octree();
        t->device = ctx->device; t->ctx = ctx; t->cfg = *cfg;
        setRootMap(t->cfg, t->map);
        st = buildOctree(*t, o, dp);
        if (st != HPSDF_OK) { delete t; return st; }
        *out = t;
        return HPSDF_OK;
    }

    HPSDF_API hpsdf_status hpsdf_query(const hpsdf_octree* tree, const double* xyz, size_t n, double* out)
    {
        if (!tree || (n && (!xyz || !out))) { setLastError("null pointer"); return HPSDF_ERR_INVALID_ARG; }
        return queryHost(*const_cast<hpsdf_octree*>(tree), xyz, n, out);
    }

    HPSDF_API hpsdf_status hpsdf_query_device(const hpsdf_octree* tree, const double* d_xyz, size_t n, double* d_out, void* stream)
    {
        if (!tree || (n && (!d_xyz || !d_out))) { setLastError("null pointer"); return HPSDF_ERR_INVALID_ARG; }
        // the kernel reads the tree's device pointers: it must run on the tree's device (the caller's stream belongs to it)
        int cur = -1;
        if (cudaGetDevice(&cur) != cudaSuccess || cur != tree->device)
        { setLastError("hpsdf_query_device: the current CUDA device is not the tree's device"); return HPSDF_ERR_INVALID_ARG; }
        HPSDF_CUDA(launchQuery(tree->view, d_xyz, n, d_out, tree->ctx->smCount, (cudaStream_t)stream));
        return HPSDF_OK;
    }

    HPSDF_API hpsdf_status hpsdf_query_with_gradient(const hpsdf_octree* tree, const double* xyz, size_t n, double* out, double* unit_grad)
    {
        if (!tree || (n && (!xyz || !out || !unit_grad))) { setLastError("null pointer"); return HPSDF_ERR_INVALID_ARG; }
        if (!n) return HPSDF_OK;
        HPSDF_CUDA(cudaSetDevice(tree->device));
        double *dIn = nullptr, *dOut = nullptr, *dG = nullptr;
        HPSDF_CUDA(cudaMalloc((void**)&dIn, n * 24));
        cudaError_t e = cudaMalloc((void**)&dOut, n * 8);
        if (e == cudaSuccess) e = cudaMalloc((void**)&dG, n * 24);
        if (e == cudaSuccess) e = cudaMemset(dG, 0, n * 24);
        if (e == cudaSuccess) e = cudaMemcpy(dIn, xyz, n * 24, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = launchQueryGradient(tree->view, dIn, n, dOut, dG, nullptr);
        if (e == cudaSuccess) e = cudaMemcpy(out, dOut, n * 8, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(unit_grad, dG, n * 24, cudaMemcpyDeviceToHost);
        cudaFree(dIn); cudaFree(dOut); cudaFree(dG);
        if (e != cudaSuccess) return failCuda(e, "hpsdf_query_with_gradient");
        return HPSDF_OK;
    }

    static hpsdf_status derivativesArgs(const hpsdf_octree* tree, const void* xyz, size_t n, const void* value, const void* grad)
    {
        if (hpsdf_device_count() == 0) { setLastError("no CUDA device available: this library has no CPU path"); return HPSDF_ERR_NO_DEVICE; }
        if (!tree || (n && (!xyz || !value || !grad))) { setLastError("null pointer"); return HPSDF_ERR_INVALID_ARG; }
        return HPSDF_OK;
    }

    HPSDF_API hpsdf_status hpsdf_query_derivatives(const hpsdf_octree* tree, const double* xyz, size_t n, double* value, double* grad,
                                                   double* hess)
    {
        hpsdf_status st = derivativesArgs(tree, xyz, n, value, grad);
        if (st != HPSDF_OK || !n) return st;
        HPSDF_CUDA(cudaSetDevice(tree->device));
        double *dIn = nullptr, *dV = nullptr, *dG = nullptr, *dH = nullptr;
        HPSDF_CUDA(cudaMalloc((void**)&dIn, n * 24));
        cudaError_t e = cudaMalloc((void**)&dV, n * 8);
        if (e == cudaSuccess) e = cudaMalloc((void**)&dG, n * 24);
        if (e == cudaSuccess && hess) e = cudaMalloc((void**)&dH, n * 48);
        if (e == cudaSuccess) e = cudaMemcpy(dIn, xyz, n * 24, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = launchQueryDerivatives(tree->view, dIn, n, dV, dG, dH, tree->ctx->smCount, nullptr);
        if (e == cudaSuccess) e = cudaMemcpy(value, dV, n * 8, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(grad, dG, n * 24, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess && hess) e = cudaMemcpy(hess, dH, n * 48, cudaMemcpyDeviceToHost);
        cudaFree(dIn); cudaFree(dV); cudaFree(dG); cudaFree(dH);
        if (e != cudaSuccess) return failCuda(e, "hpsdf_query_derivatives");
        return HPSDF_OK;
    }

    HPSDF_API hpsdf_status hpsdf_query_derivatives_device(const hpsdf_octree* tree, const double* d_xyz, size_t n, double* d_value,
                                                          double* d_grad, double* d_hess, void* stream)
    {
        hpsdf_status st = derivativesArgs(tree, d_xyz, n, d_value, d_grad);
        if (st != HPSDF_OK) return st;
        int cur = -1;
        if (cudaGetDevice(&cur) != cudaSuccess || cur != tree->device)
        { setLastError("hpsdf_query_derivatives_device: the current CUDA device is not the tree's device"); return HPSDF_ERR_INVALID_ARG; }
        HPSDF_CUDA(launchQueryDerivatives(tree->view, d_xyz, n, d_value, d_grad, d_hess, tree->ctx->smCount, (cudaStream_t)stream));
        return HPSDF_OK;
    }

    HPSDF_API hpsdf_status hpsdf_query_ray(const hpsdf_octree* tree, const double* origins, const double* directions, size_t n, double t_max,
                                           unsigned char* hit, double* t)
    {
        if (!tree || (n && (!origins || !directions || !hit || !t))) { setLastError("null pointer"); return HPSDF_ERR_INVALID_ARG; }
        if (!n) return HPSDF_OK;
        HPSDF_CUDA(cudaSetDevice(tree->device));
        double *dO = nullptr, *dD = nullptr, *dT = nullptr;
        unsigned char* dH = nullptr;
        HPSDF_CUDA(cudaMalloc((void**)&dO, n * 24));
        cudaError_t e = cudaMalloc((void**)&dD, n * 24);
        if (e == cudaSuccess) e = cudaMalloc((void**)&dT, n * 8);
        if (e == cudaSuccess) e = cudaMalloc((void**)&dH, n);
        if (e == cudaSuccess) e = cudaMemcpy(dO, origins, n * 24, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMemcpy(dD, directions, n * 24, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = launchQueryRay(tree->view, dO, dD, n, t_max, dH, dT, nullptr);
        if (e == cudaSuccess) e = cudaMemcpy(hit, dH, n, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(t, dT, n * 8, cudaMemcpyDeviceToHost);
        cudaFree(dO); cudaFree(dD); cudaFree(dT); cudaFree(dH);
        if (e != cudaSuccess) return failCuda(e, "hpsdf_query_ray");
        return HPSDF_OK;
    }

    static hpsdf_status raycastArgs(const hpsdf_octree* tree, const void* origins, const void* directions, size_t n, double t_min,
                                    double t_max, double iso, const void* t_hit, const char* fn)
    {
        if (hpsdf_device_count() == 0) { setLastError("no CUDA device available: this library has no CPU path"); return HPSDF_ERR_NO_DEVICE; }
        if (!tree || (n && (!origins || !directions || !t_hit))) { setLastError("null pointer"); return HPSDF_ERR_INVALID_ARG; }
        if (!std::isfinite(t_min) || !std::isfinite(iso) || !(t_max >= t_min))
        { setLastError(std::string(fn) + ": t_min and iso must be finite and t_max >= t_min"); return HPSDF_ERR_INVALID_ARG; }
        return HPSDF_OK;
    }

    HPSDF_API hpsdf_status hpsdf_raycast(const hpsdf_octree* tree, const double* origins, const double* directions, size_t n, double t_min,
                                         double t_max, double iso, double* t_hit, double* normals)
    {
        hpsdf_status st = raycastArgs(tree, origins, directions, n, t_min, t_max, iso, t_hit, "hpsdf_raycast");
        if (st != HPSDF_OK || !n) return st;
        HPSDF_CUDA(cudaSetDevice(tree->device));
        double *dO = nullptr, *dD = nullptr, *dT = nullptr, *dN = nullptr;
        HPSDF_CUDA(cudaMalloc((void**)&dO, n * 24));
        cudaError_t e = cudaMalloc((void**)&dD, n * 24);
        if (e == cudaSuccess) e = cudaMalloc((void**)&dT, n * 8);
        if (e == cudaSuccess && normals) e = cudaMalloc((void**)&dN, n * 24);
        if (e == cudaSuccess) e = cudaMemcpy(dO, origins, n * 24, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMemcpy(dD, directions, n * 24, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = launchRaycast(tree->view, dO, dD, n, t_min, t_max, iso, dT, dN, tree->ctx->smCount, nullptr);
        if (e == cudaSuccess) e = cudaMemcpy(t_hit, dT, n * 8, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess && normals) e = cudaMemcpy(normals, dN, n * 24, cudaMemcpyDeviceToHost);
        cudaFree(dO); cudaFree(dD); cudaFree(dT); cudaFree(dN);
        if (e != cudaSuccess) return failCuda(e, "hpsdf_raycast");
        return HPSDF_OK;
    }

    HPSDF_API hpsdf_status hpsdf_raycast_device(const hpsdf_octree* tree, const double* d_origins, const double* d_directions, size_t n,
                                                double t_min, double t_max, double iso, double* d_t_hit, double* d_normals, void* stream)
    {
        hpsdf_status st = raycastArgs(tree, d_origins, d_directions, n, t_min, t_max, iso, d_t_hit, "hpsdf_raycast_device");
        if (st != HPSDF_OK) return st;
        int cur = -1;
        if (cudaGetDevice(&cur) != cudaSuccess || cur != tree->device)
        { setLastError("hpsdf_raycast_device: the current CUDA device is not the tree's device"); return HPSDF_ERR_INVALID_ARG; }
        HPSDF_CUDA(launchRaycast(tree->view, d_origins, d_directions, n, t_min, t_max, iso, d_t_hit, d_normals, tree->ctx->smCount,
                                 (cudaStream_t)stream));
        return HPSDF_OK;
    }

    HPSDF_API hpsdf_status hpsdf_extract_isosurface(const hpsdf_octree* tree, const uint32_t resolution[3], const double box_min[3],
                                                    const double box_max[3], double iso, size_t* n_vertices, float** vertices,
                                                    size_t* n_triangles, uint32_t** tri_indices)
    {
        if (hpsdf_device_count() == 0) { setLastError("no CUDA device available: this library has no CPU path"); return HPSDF_ERR_NO_DEVICE; }
        if (!tree || !resolution || !n_vertices || !vertices || !n_triangles || !tri_indices) { setLastError("null pointer"); return HPSDF_ERR_INVALID_ARG; }
        *n_vertices = 0; *vertices = nullptr; *n_triangles = 0; *tri_indices = nullptr;
        if (!box_min != !box_max) { setLastError("hpsdf_extract_isosurface: give both box corners or neither"); return HPSDF_ERR_INVALID_ARG; }
        IsoGrid g;
        g.iso = iso;
        for (int a = 0; a < 3; ++a)
        {
            if (resolution[a] < 1 || resolution[a] > 1024) { setLastError("hpsdf_extract_isosurface: resolution outside [1, 1024]"); return HPSDF_ERR_INVALID_ARG; }
            const double lo = box_min ? box_min[a] : (double)tree->cfg.root_min[a], hi = box_max ? box_max[a] : (double)tree->cfg.root_max[a];
            if (!(lo < hi) || !std::isfinite(lo) || !std::isfinite(hi)) { setLastError("hpsdf_extract_isosurface: the box needs finite min < max"); return HPSDF_ERR_INVALID_ARG; }
            g.n[a] = resolution[a];
            g.lo[a] = lo;
            g.h[a] = (hi - lo) / (double)resolution[a];
        }
        const uint32_t nPoints = (g.n[0] + 1) * (g.n[1] + 1) * (g.n[2] + 1);        // <= 1025^3 < 2^32
        HPSDF_CUDA(cudaSetDevice(tree->device));
        // HPSDF_ISO_TIMES: device time of the phases on stderr (grid, count + scans, emit, copy)
        const bool timed = getenv("HPSDF_ISO_TIMES") != nullptr;
        cudaStream_t stream = nullptr;
        cudaEvent_t ev[6] = { nullptr, nullptr, nullptr, nullptr, nullptr, nullptr };
        void* scratch = nullptr;
        char* dOut = nullptr;
        float* hV = nullptr;
        uint32_t* hT = nullptr;
        unsigned long long totals[2] = { 0, 0 };
        hpsdf_status st = HPSDF_OK;
        cudaError_t e = cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking);
        for (int i = 0; i < 6 && timed && e == cudaSuccess; ++i) e = cudaEventCreate(&ev[i]);
        auto mark = [&](int i) { if (timed && e == cudaSuccess) e = cudaEventRecord(ev[i], stream); };
        if (e == cudaSuccess) e = cudaMalloc(&scratch, isoScratchBytes(nPoints));
        IsoScratch s{};
        if (e == cudaSuccess) s = carveIsoScratch(scratch, nPoints);
        mark(0);
        if (e == cudaSuccess) e = launchIsoGrid(tree->view, g, s, tree->ctx->smCount, stream);
        mark(1);
        if (e == cudaSuccess) e = launchIsoCount(g, s, tree->ctx->smCount, totals, stream);
        mark(2);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        const size_t nv = (size_t)totals[0], nt = (size_t)totals[1];
        if (e == cudaSuccess && (totals[0] > 0xFFFFFFFFull || totals[1] > 0xFFFFFFFFull))
        {
            setLastError("hpsdf_extract_isosurface: " + std::to_string(totals[0]) + " vertices and " + std::to_string(totals[1]) +
                         " triangles: a count above 2^32 - 1 does not fit the uint32 indices");
            st = HPSDF_ERR_UNSUPPORTED;
        }
        const size_t vBytes = (nv * 12 + 255) & ~(size_t)255;
        if (e == cudaSuccess && st == HPSDF_OK && nv)
        {
            e = cudaMalloc((void**)&dOut, vBytes + nt * 12);
            hV = (float*)malloc(nv * 12);
            hT = (uint32_t*)malloc(nt * 12);
            if (e == cudaSuccess && (!hV || !hT)) { setLastError("hpsdf_extract_isosurface: host allocation failed"); st = HPSDF_ERR_OOM; }
            mark(3);
            if (e == cudaSuccess && st == HPSDF_OK) e = launchIsoEmit(g, s, (float*)dOut, (uint32_t*)(dOut + vBytes), stream);
            mark(4);
            if (e == cudaSuccess && st == HPSDF_OK) e = cudaMemcpyAsync(hV, dOut, nv * 12, cudaMemcpyDeviceToHost, stream);
            if (e == cudaSuccess && st == HPSDF_OK) e = cudaMemcpyAsync(hT, dOut + vBytes, nt * 12, cudaMemcpyDeviceToHost, stream);
            mark(5);
            if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        }
        if (timed && e == cudaSuccess && st == HPSDF_OK)
        {
            float ms[4] = { 0, 0, 0, 0 };
            cudaEventElapsedTime(&ms[0], ev[0], ev[1]);
            cudaEventElapsedTime(&ms[1], ev[1], ev[2]);
            if (nv) { cudaEventElapsedTime(&ms[2], ev[3], ev[4]); cudaEventElapsedTime(&ms[3], ev[4], ev[5]); }
            fprintf(stderr, "hpsdf_extract_isosurface: %u x %u x %u cells, %zu vertices, %zu triangles; grid %.3f ms, count+scan %.3f ms, emit %.3f ms, copy %.3f ms\n",
                    g.n[0], g.n[1], g.n[2], nv, nt, ms[0], ms[1], ms[2], ms[3]);
        }
        if (stream) cudaStreamSynchronize(stream);
        for (int i = 0; i < 6; ++i) if (ev[i]) cudaEventDestroy(ev[i]);
        if (stream) cudaStreamDestroy(stream);
        cudaFree(scratch);
        cudaFree(dOut);
        if (e != cudaSuccess) st = failCuda(e, "hpsdf_extract_isosurface");
        if (st != HPSDF_OK) { free(hV); free(hT); return st; }
        *n_vertices = nv; *vertices = hV; *n_triangles = nt; *tri_indices = hT;
        return HPSDF_OK;
    }

    HPSDF_API hpsdf_status hpsdf_to_memory_block(const hpsdf_octree* tree, size_t* size, void** ptr)
    {
        if (!tree || !size || !ptr) { setLastError("null pointer"); return HPSDF_ERR_INVALID_ARG; }
        return toMemoryBlock(*tree, size, ptr);
    }

    HPSDF_API hpsdf_status hpsdf_from_memory_block(const void* ptr, size_t size, int device, hpsdf_octree** out)
    {
        if (!out) { setLastError("out is null"); return HPSDF_ERR_INVALID_ARG; }
        *out = nullptr;
        if (!ptr || !size) { setLastError("MemoryBlock is null or empty"); return HPSDF_ERR_BAD_BLOCK; }   // Octree.cpp:405
        DeviceCtx* ctx = nullptr;
        hpsdf_status st = needDevice(device, &ctx);
        if (st != HPSDF_OK) return st;
        hpsdf_octree* t = new hpsdf_octree();
        t->device = ctx->device; t->ctx = ctx;
        st = fromMemoryBlock(*t, ptr, size);
        if (st != HPSDF_OK) { delete t; return st; }
        *out = t;
        return HPSDF_OK;
    }

    // Octree copy constructor (Octree.cpp:24-45): nodes, config and the coefficient store are duplicated.
    HPSDF_API hpsdf_status hpsdf_clone(const hpsdf_octree* tree, hpsdf_octree** out)
    {
        if (!tree || !out) { setLastError("null pointer"); return HPSDF_ERR_INVALID_ARG; }
        *out = nullptr;
        HPSDF_CUDA(cudaSetDevice(tree->device));
        hpsdf_octree* src = const_cast<hpsdf_octree*>(tree);
        hpsdf_status hs = ensureHostNodes(*src);
        if (hs != HPSDF_OK) return hs;
        ensureDecisionLog(*src);
        ensureApplyLog(*src);
        hpsdf_octree* t = new hpsdf_octree();
        t->device = tree->device; t->ctx = tree->ctx; t->cfg = tree->cfg; t->map = tree->map;
        t->nodes = tree->nodes; t->nNodes = tree->nNodes; t->nCoeffs = tree->nCoeffs; t->nCoeffsPad = tree->nCoeffsPad;
        t->stats = tree->stats; t->decisionLog = tree->decisionLog; t->applyLog = tree->applyLog;
        hpsdf_status st = allocTreeBlob(*t);
        if (st != HPSDF_OK) { delete t; return st; }
        cudaError_t e = cudaMemcpy(t->dCoeffs, tree->dCoeffs, t->nCoeffs * 8, cudaMemcpyDeviceToDevice);
        if (e != cudaSuccess) { delete t; return failCuda(e, "hpsdf_clone"); }
        std::lock_guard<std::mutex> wsLock(*(std::mutex*)t->ctx->wsMutex);
        st = finalizeQueryStructures(*t, t->ctx->ws.stream);
        if (st != HPSDF_OK) { delete t; return st; }
        *out = t;
        return HPSDF_OK;
    }

    HPSDF_API hpsdf_status hpsdf_get_root_aabb(const hpsdf_octree* tree, float mn[3], float mx[3])
    {
        if (!tree || !mn || !mx) { setLastError("null pointer"); return HPSDF_ERR_INVALID_ARG; }
        memcpy(mn, tree->cfg.root_min, 12); memcpy(mx, tree->cfg.root_max, 12);     // Octree.cpp:106-109: config.root
        return HPSDF_OK;
    }

    HPSDF_API hpsdf_status hpsdf_get_config(const hpsdf_octree* tree, hpsdf_config* cfg)
    {
        if (!tree || !cfg) { setLastError("null pointer"); return HPSDF_ERR_INVALID_ARG; }
        *cfg = tree->cfg;
        return HPSDF_OK;
    }

    HPSDF_API hpsdf_status hpsdf_get_device(const hpsdf_octree* tree, int* device)
    {
        if (!tree || !device) { setLastError("null pointer"); return HPSDF_ERR_INVALID_ARG; }
        *device = tree->device;
        return HPSDF_OK;
    }

    HPSDF_API void hpsdf_destroy(hpsdf_octree* tree) { delete tree; }

    HPSDF_API hpsdf_status hpsdf_get_build_stats(const hpsdf_octree* tree, hpsdf_build_stats* stats)
    {
        if (!tree || !stats) { setLastError("null pointer"); return HPSDF_ERR_INVALID_ARG; }
        *stats = tree->stats;
        return HPSDF_OK;
    }

    HPSDF_API size_t hpsdf_get_decision_log(const hpsdf_octree* tree, hpsdf_decision_log_entry* out, size_t capacity)
    {
        if (!tree) return 0;
        ensureDecisionLog(*const_cast<hpsdf_octree*>(tree));
        const size_t n = tree->decisionLog.size();
        if (out) memcpy(out, tree->decisionLog.data(), std::min(n, capacity) * sizeof(hpsdf_decision_log_entry));
        return n;
    }

    HPSDF_API size_t hpsdf_get_apply_log(const hpsdf_octree* tree, hpsdf_apply_log_entry* out, size_t capacity)
    {
        if (!tree) return 0;
        ensureApplyLog(*const_cast<hpsdf_octree*>(tree));
        const size_t n = tree->applyLog.size();
        if (out) memcpy(out, tree->applyLog.data(), std::min(n, capacity) * sizeof(hpsdf_apply_log_entry));
        return n;
    }

    HPSDF_API void hpsdf_set_jit(int on) { setJitDefault(on != 0); }

    HPSDF_API hpsdf_status hpsdf_jit_compile_check(const hpsdf_sdf_program* prog, uint32_t degree, char* source_out, size_t source_cap, size_t* cubin_bytes)
    {
        if (degree < 1 || degree > (uint32_t)kMaxDegree) { setLastError("bad degree"); return HPSDF_ERR_INVALID_ARG; }
        SdfProgramDev dp;
        hpsdf_status st = resolveProgram(prog, -1, dp);
        if (st != HPSDF_OK) return st;
        std::string src, why;
        const bool ok = jitCompileCheck(dp, (int)degree, &src, cubin_bytes, why);
        if (source_out && source_cap) { const size_t k = std::min(source_cap - 1, src.size()); memcpy(source_out, src.data(), k); source_out[k] = 0; }
        if (!ok) { setLastError("JIT fit kernel: " + why); return HPSDF_ERR_UNSUPPORTED; }
        return HPSDF_OK;
    }

    HPSDF_API hpsdf_status hpsdf_fit_batch(const hpsdf_config* cfg, const hpsdf_sdf_program* prog, const float* cells, const uint8_t* depth,
                                           size_t n, uint32_t degree, double* coeffs_out, double* raw_err_out, int device, float* elapsed_ms)
    {
        if (!cfg || !cells || !depth || !coeffs_out || !raw_err_out || degree < 1 || degree > (uint32_t)kMaxDegree - 1)
        { setLastError("bad hpsdf_fit_batch arguments"); return HPSDF_ERR_INVALID_ARG; }
        DeviceCtx* ctx = nullptr;
        hpsdf_status st = needDevice(device, &ctx);
        if (st != HPSDF_OK) return st;
        SdfProgramDev dp;
        if ((st = resolveProgram(prog, ctx->device, dp)) != HPSDF_OK) return st;
        if (!n) return HPSDF_OK;
        for (size_t i = 0; i < n; ++i)            // c_nl has kMaxDepth + 1 columns; a cell needs a positive size
            if (depth[i] > (uint8_t)kMaxDepth || !(cells[4 * i + 3] > 0.0f))
            { setLastError("hpsdf_fit_batch: depth above TREE_MAX_DEPTH or non-positive half size"); return HPSDF_ERR_INVALID_ARG; }
        RootMap map;
        setRootMap(*cfg, map);
        const size_t nc = (size_t)coeffCount((int)degree);
        if (n * nc >= 0xFFFFFFF0ull) { setLastError("batch too large"); return HPSDF_ERR_INVALID_ARG; }
        std::vector<FitTask> tasks(n);
        for (size_t i = 0; i < n; ++i)
        {
            FitTask& t = tasks[i];
            t.cx = cells[4 * i]; t.cy = cells[4 * i + 1]; t.cz = cells[4 * i + 2]; t.half = cells[4 * i + 3];
            t.out = (uint32_t)(i * nc); t.src = kNoSrc; t.depth = depth[i]; t.degree = (uint8_t)degree; t.degreeIn = 0; t.pad = 0; t.rec = (uint32_t)i;
        }
        FitTask* dT = nullptr; double* dPool = nullptr; FitRecord* dR = nullptr;
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        cudaError_t e = cudaMalloc((void**)&dT, n * sizeof(FitTask));
        if (e == cudaSuccess) e = cudaMalloc((void**)&dPool, n * nc * 8);
        if (e == cudaSuccess) e = cudaMalloc((void**)&dR, n * sizeof(FitRecord));
        if (e == cudaSuccess) e = cudaMemcpy(dT, tasks.data(), n * sizeof(FitTask), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaEventCreate(&e0);
        if (e == cudaSuccess) e = cudaEventCreate(&e1);
        if (e == cudaSuccess) e = cudaEventRecord(e0, nullptr);
        hpsdf_status ls = HPSDF_OK;
        std::unique_lock<std::mutex> wsLock(*(std::mutex*)ctx->wsMutex);      // the sample scratch of mesh / octree programs is per device
        if (e == cudaSuccess) ls = launchFit(0, (int)degree, dT, (int)n, dPool, dR, dp, map, *ctx, nullptr);
        if (e == cudaSuccess) e = cudaEventRecord(e1, nullptr);
        if (e == cudaSuccess) e = cudaMemcpy(coeffs_out, dPool, n * nc * 8, cudaMemcpyDeviceToHost);
        std::vector<FitRecord> recs(n);
        if (e == cudaSuccess) e = cudaMemcpy(recs.data(), dR, n * sizeof(FitRecord), cudaMemcpyDeviceToHost);
        if (e == cudaSuccess && elapsed_ms) e = cudaEventElapsedTime(elapsed_ms, e0, e1);
        if (getenv("HPSDF_MESH_STATS")) printMeshStats();
        if (e == cudaSuccess) for (size_t i = 0; i < n; ++i) raw_err_out[i] = recs[i].rawErr;
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
        cudaFree(dT); cudaFree(dPool); cudaFree(dR);
        if (e != cudaSuccess) return failCuda(e, "hpsdf_fit_batch");
        return ls;
    }

    // Synthetic frontier (SURVEY.md §8d): all cells of a uniform grid at grid_depth as refinement jobs at degree p:
    // 8 child fits @p (depth+1, from scratch) + 1 p-fit @p+1 (shell only, lower shells copied from a zero slot).
    HPSDF_API hpsdf_status hpsdf_bench_frontier(const hpsdf_config* cfg, const hpsdf_sdf_program* prog, uint32_t grid_depth, uint32_t degree,
                                                uint32_t repeats, int device, void* stream_, hpsdf_frontier_bench* out)
    {
        if (!cfg || !out || grid_depth < 1 || grid_depth > 7 || degree < 2 || degree > (uint32_t)kMaxDegree - 2 || repeats < 1)
        { setLastError("bad hpsdf_bench_frontier arguments"); return HPSDF_ERR_INVALID_ARG; }
        DeviceCtx* ctx = nullptr;
        hpsdf_status st = needDevice(device, &ctx);
        if (st != HPSDF_OK) return st;
        SdfProgramDev dp;
        if ((st = resolveProgram(prog, ctx->device, dp)) != HPSDF_OK) return st;
        RootMap map;
        setRootMap(*cfg, map);
        cudaStream_t stream = (cudaStream_t)stream_;
        const uint32_t g = 1u << grid_depth;
        const size_t jobs = (size_t)g * g * g;
        const size_t ncH = coeffCount((int)degree), ncP = coeffCount((int)degree + 1);
        const size_t nH = 8 * jobs, nP = jobs;
        if (nH * ncH + nP * ncP + ncP >= 0xFFFFFFF0ull) { setLastError("frontier too large"); return HPSDF_ERR_INVALID_ARG; }
        std::vector<FitTask> tasks(nH + nP);
        const float cell = 1.0f / (float)g;
        size_t ti = 0;
        const uint32_t zeroSlot = 0;              // ncP zeros at the start of the pool: the "existing" coefficients of the p-fits
        size_t poolCur = ncP;
        for (uint32_t z = 0; z < g; ++z) for (uint32_t y = 0; y < g; ++y) for (uint32_t x = 0; x < g; ++x)
            for (uint32_t c = 0; c < 8; ++c)
            {
                FitTask& t = tasks[ti];
                const float cx = -0.5f + cell * ((float)x + 0.5f), cy = -0.5f + cell * ((float)y + 0.5f), cz = -0.5f + cell * ((float)z + 0.5f);
                t.half = cell * 0.25f;
                t.cx = cx + ((c & 1) ? t.half : -t.half); t.cy = cy + ((c & 2) ? t.half : -t.half); t.cz = cz + ((c & 4) ? t.half : -t.half);
                t.out = (uint32_t)poolCur; poolCur += ncH; t.src = kNoSrc;
                t.depth = (uint8_t)std::min<uint32_t>(grid_depth + 1, kMaxDepth); t.degree = (uint8_t)degree; t.degreeIn = 0; t.pad = 0; t.rec = (uint32_t)ti;
                ++ti;
            }
        for (uint32_t z = 0; z < g; ++z) for (uint32_t y = 0; y < g; ++y) for (uint32_t x = 0; x < g; ++x)
        {
            FitTask& t = tasks[ti];
            t.cx = -0.5f + cell * ((float)x + 0.5f); t.cy = -0.5f + cell * ((float)y + 0.5f); t.cz = -0.5f + cell * ((float)z + 0.5f);
            t.half = cell * 0.5f;
            t.out = (uint32_t)poolCur; poolCur += ncP; t.src = zeroSlot;
            t.depth = (uint8_t)grid_depth; t.degree = (uint8_t)(degree + 1); t.degreeIn = (uint8_t)degree; t.pad = 0; t.rec = (uint32_t)ti;
            ++ti;
        }
        FitTask* dT = nullptr; double* dPool = nullptr; FitRecord* dR = nullptr;
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        cudaError_t e = cudaMalloc((void**)&dT, tasks.size() * sizeof(FitTask));
        if (e == cudaSuccess) e = cudaMalloc((void**)&dPool, poolCur * 8);
        if (e == cudaSuccess) e = cudaMalloc((void**)&dR, tasks.size() * sizeof(FitRecord));
        if (e == cudaSuccess) e = cudaMemsetAsync(dPool, 0, ncP * 8, stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(dT, tasks.data(), tasks.size() * sizeof(FitTask), cudaMemcpyHostToDevice, stream);
        if (e == cudaSuccess) e = cudaEventCreate(&e0);
        if (e == cudaSuccess) e = cudaEventCreate(&e1);
        hpsdf_status ls = HPSDF_OK;
        std::unique_lock<std::mutex> wsLock(*(std::mutex*)ctx->wsMutex);
        for (uint32_t r = 0; r <= repeats && e == cudaSuccess && ls == HPSDF_OK; ++r)
        {
            if (r == 1) e = cudaEventRecord(e0, stream);          // launch 0 is the warm-up
            if (e == cudaSuccess && ls == HPSDF_OK) ls = launchFit(0, (int)degree, dT, (int)nH, dPool, dR, dp, map, *ctx, stream);
            if (e == cudaSuccess && ls == HPSDF_OK) ls = launchFit(0, (int)degree + 1, dT + nH, (int)nP, dPool, dR, dp, map, *ctx, stream);
        }
        if (e == cudaSuccess) e = cudaEventRecord(e1, stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        float ms = 0.0f;
        if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
        std::vector<FitRecord> recs(tasks.size());
        if (e == cudaSuccess) e = cudaMemcpy(recs.data(), dR, recs.size() * sizeof(FitRecord), cudaMemcpyDeviceToHost);
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
        cudaFree(dT); cudaFree(dPool); cudaFree(dR);
        if (e != cudaSuccess) return failCuda(e, "hpsdf_bench_frontier");
        if (ls != HPSDF_OK) return ls;
        memset(out, 0, sizeof(*out));
        out->ms_per_launch = (double)ms / repeats;
        out->jobs = jobs; out->fits = nH + nP;
        const uint64_t nh = fitRule((int)degree), np = fitRule((int)degree + 1);
        out->sdf_evals = nH * nh * nh * nh + nP * np * np * np;
        const double cF = summarizeProgram(dp).flopsPerEval;
        out->sdf_flops_per_eval = cF;
        out->algorithmic_flops = (double)nH * fitFlops((int)degree) + (double)nP * fitFlops((int)degree + 1) + cF * (double)out->sdf_evals;
        for (const FitRecord& r : recs) out->checksum += r.rawErr;
        return HPSDF_OK;
    }

    HPSDF_API hpsdf_status hpsdf_uniform_points_device(uint64_t seed, uint64_t first_index, size_t n, const double lo[3], const double hi[3],
                                                       double* d_xyz, void* stream)
    {
        if (n && (!lo || !hi || !d_xyz)) { setLastError("null pointer"); return HPSDF_ERR_INVALID_ARG; }
        if (hpsdf_device_count() == 0) { setLastError("no CUDA device available: this library has no CPU path"); return HPSDF_ERR_NO_DEVICE; }
        HPSDF_CUDA(launchUniformPoints(seed, first_index, n, lo, hi, d_xyz, (cudaStream_t)stream));
        return HPSDF_OK;
    }

    HPSDF_API hpsdf_status hpsdf_measure_fp64_peak(int device, void* stream_, double* tflops)
    {
        if (!tflops) { setLastError("null pointer"); return HPSDF_ERR_INVALID_ARG; }
        DeviceCtx* ctx = nullptr;
        hpsdf_status st = needDevice(device, &ctx);
        if (st != HPSDF_OK) return st;
        cudaStream_t stream = (cudaStream_t)stream_;
        const int blocks = ctx->smCount * 8;
        double* dOut = nullptr;
        HPSDF_CUDA(cudaMalloc((void**)&dOut, (size_t)blocks * 256 * 8));
        cudaEvent_t e0, e1;
        cudaEventCreate(&e0); cudaEventCreate(&e1);
        cudaError_t e = launchDfmaPeak(dOut, blocks, stream);      // warm-up
        double best = 0.0;
        for (int r = 0; r < 5 && e == cudaSuccess; ++r)
        {
            cudaEventRecord(e0, stream);
            for (int k = 0; k < 4 && e == cudaSuccess; ++k) e = launchDfmaPeak(dOut, blocks, stream);
            cudaEventRecord(e1, stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
            float ms = 0.0f;
            cudaEventElapsedTime(&ms, e0, e1);
            const double flops = 4.0 * (double)blocks * 256.0 * 512.0 * 8.0 * 8.0 * 2.0;
            if (ms > 0.0f) best = std::max(best, flops / (ms * 1e-3) / 1e12);
        }
        cudaEventDestroy(e0); cudaEventDestroy(e1);
        cudaFree(dOut);
        if (e != cudaSuccess) return failCuda(e, "hpsdf_measure_fp64_peak");
        *tflops = best;
        return HPSDF_OK;
    }

}
