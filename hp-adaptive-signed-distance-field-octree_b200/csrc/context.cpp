// context.cpp — per-device context: projection tables uploaded once, error plumbing, small helpers.
#include <chrono>
#include <cstring>
#include <mutex>
#include <vector>
#include "octree.h"

namespace hpsdf
{
    namespace
    {
        thread_local std::string g_lastError;
        std::mutex g_ctxMutex;
        DeviceCtx* g_ctx[16] = { nullptr };

        // P_a(x) by the three-term recurrence with the reference's precomputed constants (LpX, Octree.cpp:988-1004)
        double legendre(int a, double x)
        {
            const Tables& t = tables();
            double m2 = 0.0, m1 = 1.0, l = 1.0;
            for (int i = 1; i <= a; ++i) { l = t.rec[i][0] * x * m1 - t.rec[i][1] * m2; m2 = m1; m1 = l; }
            return l;
        }
    }

    void setLastError(const std::string& msg) { g_lastError = msg; }
    const std::string& lastError() { return g_lastError; }

    hpsdf_status failCuda(cudaError_t e, const char* what)
    {
        setLastError(std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what);
        cudaGetLastError();   // clear the sticky flag of non-fatal errors
        return (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) ? HPSDF_ERR_NO_DEVICE
             : (e == cudaErrorMemoryAllocation) ? HPSDF_ERR_OOM : HPSDF_ERR_CUDA;
    }

    double nowMs()
    {
        return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
    }

    struct BlobCache
    {
        std::mutex m;
        std::vector<std::pair<void*, size_t>> free;
        size_t bytes = 0;
    };

    cudaError_t acquireBlob(DeviceCtx& ctx, size_t bytes, void** ptr, size_t* capacity)
    {
        BlobCache& c = *(BlobCache*)ctx.blobCache;
        const size_t want = (bytes + ((size_t)1 << 20) - 1) & ~(((size_t)1 << 20) - 1);
        {
            std::lock_guard<std::mutex> lock(c.m);
            int best = -1;
            for (int i = 0; i < (int)c.free.size(); ++i)
                if (c.free[i].second >= want && c.free[i].second <= 4 * want && (best < 0 || c.free[i].second < c.free[best].second)) best = i;
            if (best >= 0)
            {
                *ptr = c.free[best].first; *capacity = c.free[best].second;
                c.bytes -= c.free[best].second;
                c.free.erase(c.free.begin() + best);
                return cudaSuccess;
            }
        }
        *capacity = want;
        return cudaMalloc(ptr, want);
    }

    void releaseBlob(DeviceCtx& ctx, void* ptr, size_t capacity)
    {
        if (!ptr) return;
        BlobCache& c = *(BlobCache*)ctx.blobCache;
        {
            std::lock_guard<std::mutex> lock(c.m);
            if (c.free.size() < 8 && c.bytes + capacity <= ((size_t)2 << 30))
            {
                c.free.emplace_back(ptr, capacity);
                c.bytes += capacity;
                return;
            }
        }
        cudaFree(ptr);
    }

    DeviceCtx* getDeviceCtx(int device, std::string& err)
    {
        std::lock_guard<std::mutex> lock(g_ctxMutex);
        int count = 0;
        cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess || count == 0)
        {
            cudaGetLastError();
            err = "no CUDA device available: this library has no CPU path";
            return nullptr;
        }
        if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) device = 0; }
        if (device >= count || device >= 16) { err = "device ordinal out of range"; return nullptr; }
        if (g_ctx[device]) { cudaSetDevice(device); return g_ctx[device]; }
        if ((e = cudaSetDevice(device)) != cudaSuccess) { err = cudaGetErrorString(e); return nullptr; }

        // Layout of the table buffer: per degree d = 1..12: q[(d+1)*n] then roots[n]; then bidx[455] (uint32).
        std::vector<double> host;
        size_t qOff[kMaxDegree + 1] = { 0 }, rOff[kMaxDegree + 1] = { 0 };
        for (int d = 1; d <= kMaxDegree; ++d)
        {
            const int n = fitRule(d);
            const double* r = glRoots(n);
            const double* w = glWeights(n);
            qOff[d] = host.size();
            for (int c = 0; c <= d; ++c)
                for (int k = 0; k < n; ++k) host.push_back(w[k] * legendre(c, r[k]));
            rOff[d] = host.size();
            for (int k = 0; k < n; ++k) host.push_back(r[k]);
        }
        const size_t glOff = host.size();
        for (int i = 0; i < 2080; ++i) host.push_back(glRoots(1)[i]);
        for (int i = 0; i < 2080; ++i) host.push_back(glWeights(1)[i]);
        const size_t bidxOff = host.size();
        std::vector<uint32_t> bidx(kMaxCoeffs + 1, 0);
        for (int i = 0; i < kMaxCoeffs; ++i)
            bidx[i] = (uint32_t)tables().bidx[i][0] | ((uint32_t)tables().bidx[i][1] << 8) | ((uint32_t)tables().bidx[i][2] << 16);
        const size_t bytes = host.size() * sizeof(double) + bidx.size() * sizeof(uint32_t);
        void* mem = nullptr;
        if ((e = cudaMalloc(&mem, bytes)) != cudaSuccess) { err = cudaGetErrorString(e); return nullptr; }
        cudaMemcpy(mem, host.data(), host.size() * sizeof(double), cudaMemcpyHostToDevice);
        cudaMemcpy((char*)mem + bidxOff * sizeof(double), bidx.data(), bidx.size() * sizeof(uint32_t), cudaMemcpyHostToDevice);

        DeviceCtx* ctx = new DeviceCtx();
        ctx->device = device;
        ctx->tabMem = mem;
        const double* base = (const double*)mem;
        for (int d = 0; d <= kMaxDegree; ++d)
        {
            ctx->fitTab.q[d]     = d ? base + qOff[d] : nullptr;
            ctx->fitTab.roots[d] = d ? base + rOff[d] : nullptr;
        }
        ctx->fitTab.bidx = (const uint32_t*)(base + bidxOff);
        ctx->glRoots = base + glOff; ctx->glWeights = base + glOff + 2080;
        cudaDeviceGetAttribute(&ctx->smCount, cudaDevAttrMultiProcessorCount, device);
        uploadConstants();
        ctx->wsMutex = new std::mutex();
        ctx->blobCache = new BlobCache();
        cudaStreamCreateWithFlags(&ctx->ws.stream, cudaStreamNonBlocking);
        cudaEventCreate(&ctx->ws.ev0);
        cudaEventCreate(&ctx->ws.ev1);
        cudaEventCreateWithFlags(&ctx->ws.evFork, cudaEventDisableTiming);
        for (int i = 0; i < 4; ++i)
        {
            cudaStreamCreateWithFlags(&ctx->ws.aux[i], cudaStreamNonBlocking);
            cudaEventCreateWithFlags(&ctx->ws.evJoin[i], cudaEventDisableTiming);
        }
        // a first pool of 32 M doubles (256 MB) and pinned staging for 128 K fits: a README-sized build never reallocates
        ctx->ws.pool.reserve((size_t)32 << 20);
        ctx->ws.tasks.reserve((size_t)1 << 17); ctx->ws.recs.reserve((size_t)1 << 17);
        ctx->ws.hRecs.reserve((size_t)1 << 17);
        if ((e = cudaDeviceSynchronize()) != cudaSuccess) { err = cudaGetErrorString(e); delete ctx; cudaFree(mem); return nullptr; }
        g_ctx[device] = ctx;
        return ctx;
    }

    void setRootMap(const hpsdf_config& cfg, RootMap& map)
    {
        // Octree.cpp:322-324 / 419-420: centre, sizes and 1/size are computed in f32, then widened.
        for (int i = 0; i < 3; ++i)
        {
            const float c = (cfg.root_min[i] + cfg.root_max[i]) / 2.0f;
            const float s = cfg.root_max[i] - cfg.root_min[i];
            map.centre[i]   = (double)c;
            map.sizes[i]    = (double)s;
            map.invSizes[i] = (double)(1.0f / s);
        }
    }

    void cornerAabb(const HostNode& p, uint32_t i, float mn[3], float mx[3])
    {
        for (int d = 0; d < 3; ++d)
        {
            const float mid = (p.mx[d] + p.mn[d]) * 0.5f;
            mn[d] = (i & (1u << d)) ? mid : p.mn[d];
            mx[d] = (i & (1u << d)) ? p.mx[d] : mid;
        }
    }
}
