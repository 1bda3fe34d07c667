// mesh.cpp — device-resident triangle mesh as an SDF source: what replaces Meshing::Mesh + Meshing::BVH
// (Include/Meshing/Mesh.h, Include/Meshing/BVH.h) under Octree::Create.
//
// hpsdf_mesh_create uploads the vertex / index arrays and runs the whole set-up as kernels (mesh_build.cuh): half-edge twins
// (Mesh::CreateHalfEdges, Source/Meshing/Mesh.cpp:87-131; an unpaired edge -> HPSDF_ERR_MESH), float32 pseudonormals with the
// reference's formulas and operation order (Mesh.cpp:185-242), a median-split BVH with oriented boxes and its 4-wide
// collapse. The host only derives the SHAPE of the tree (node count, depth — functions of the triangle count) and reads back
// two flags and the root bounds. Traversal: mesh_eval.cuh, mesh_sample_kernel.cuh.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <map>
#include <mutex>
#include <numeric>
#include <vector>
#include "octree.h"

struct hpsdf_mesh
{
    int      device = 0;
    hpsdf::DeviceCtx* ctx = nullptr;
    void*    blob = nullptr;                  // nodes | triVerts | pseudo | oriented boxes | wide nodes | view (from the device's blob cache)
    size_t   blobBytes = 0;
    hpsdf::DeviceMeshView  view{};
    hpsdf::DeviceMeshView* dView = nullptr;
    float    mn[3] = { 0, 0, 0 }, mx[3] = { 0, 0, 0 };
    uint32_t nTris = 0, nVerts = 0;
};

namespace hpsdf
{
    cudaError_t launchMeshDistance(const DeviceMeshView* dView, const float* dXyz, size_t n, float* dOut, cudaStream_t stream);   // kernels.cu

    const DeviceMeshView* meshDeviceView(const hpsdf_mesh* m) { return m ? m->dView : nullptr; }
    int meshDevice(const hpsdf_mesh* m) { return m ? m->device : -1; }

    // kernels.cu (mesh_build.cuh)
    struct MeshBuildIn { const float* v; const uint32_t* tri; uint32_t nVerts, nTris; };
    struct BvhCountTable { uint32_t n; uint32_t size[96]; uint32_t count[96]; };
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
    size_t        meshBuildTempBytes(uint32_t nTris, uint32_t nNodes);
    MeshBuildTemp carveMeshTemp(char* arena, uint32_t nTris, uint32_t nNodes);
    cudaError_t   meshBuildHalfEdgesAndPseudo(const MeshBuildIn& M, const MeshBuildTemp& T, float* pseudo, cudaStream_t stream);
    cudaError_t   meshBuildBvh(const MeshBuildIn& M, const MeshBuildTemp& T, const BvhCountTable& counts, uint32_t levels, uint32_t nNodes,
                               float* pseudo, BvhNode* nodes, const uint32_t** orderOut, cudaStream_t stream);
    cudaError_t   meshBuildBoxes(const MeshBuildIn& M, const MeshBuildTemp& T, const uint32_t* order, uint32_t nNodes, double inflate,
                                 const BvhNode* nodes, float* obb, float* wide, float4* triVerts, cudaStream_t stream);

    namespace
    {
        // The median-split tree over m triangles (leaf <= 4) is fixed by m alone: node count, depth, number of 4-wide nodes
        // (internal nodes at even depth), and the table of (size -> node count) for the sizes that occur (two per level).
        struct TreeShape
        {
            std::map<uint32_t, uint32_t> count, depth;
            std::map<std::pair<uint32_t, uint32_t>, uint32_t> wide;
            uint32_t nodes(uint32_t m)
            {
                if (m <= 4) return 1u;
                auto it = count.find(m);
                if (it != count.end()) return it->second;
                const uint32_t c = 1u + nodes(m / 2) + nodes(m - m / 2);
                count[m] = c;
                return c;
            }
            uint32_t levels(uint32_t m)
            {
                if (m <= 4) return 0u;
                auto it = depth.find(m);
                if (it != depth.end()) return it->second;
                const uint32_t d = 1u + std::max(levels(m / 2), levels(m - m / 2));
                depth[m] = d;
                return d;
            }
            uint32_t wideNodes(uint32_t m, uint32_t parity)
            {
                if (m <= 4) return 0u;
                const auto key = std::make_pair(m, parity);
                auto it = wide.find(key);
                if (it != wide.end()) return it->second;
                const uint32_t w = (parity == 0 ? 1u : 0u) + wideNodes(m / 2, parity ^ 1u) + wideNodes(m - m / 2, parity ^ 1u);
                wide[key] = w;
                return w;
            }
        };
    }
}

using namespace hpsdf;

extern "C"
{
    HPSDF_API hpsdf_status hpsdf_mesh_create(const float* vertices, size_t n_vertices, const uint32_t* tri_indices, size_t n_tris,
                                             int device, hpsdf_mesh** out)
    {
        if (!out) { setLastError("out is null"); return HPSDF_ERR_INVALID_ARG; }
        *out = nullptr;
        if (!vertices || !tri_indices || n_vertices == 0 || n_tris == 0 || n_tris >= 0x10000000ull || n_vertices >= 0xFFFFFFFFull)      // leaf slots are packed into 28 bits (mesh_sample_kernel.cuh)
        { setLastError("mesh arrays are null, empty or too large"); return HPSDF_ERR_INVALID_ARG; }
        std::string err;
        DeviceCtx* ctx = getDeviceCtx(device, err);
        if (!ctx) { setLastError(err); return HPSDF_ERR_NO_DEVICE; }

        const bool dbg = getenv("HPSDF_DEBUG_MESH") != nullptr;
        double tS = nowMs();
        auto stage = [&](const char* what) { if (dbg) { cudaDeviceSynchronize(); const double t = nowMs(); fprintf(stderr, "mesh_create: %-22s %.2f ms\n", what, t - tS); tS = t; } };

        // shape of the tree (a function of the triangle count alone)
        TreeShape shape;
        const uint32_t nT = (uint32_t)n_tris, nV = (uint32_t)n_vertices;
        const uint32_t nNodes = shape.nodes(nT), levels = shape.levels(nT), nWide = std::max(1u, shape.wideNodes(nT, 0));
        // traversal stacks (mesh_eval.cuh, mesh_sample_kernel.cuh) hold 48 entries: one push per binary level, three per 4-wide level
        if (levels > 47u || 3u * ((levels + 1u) / 2u) > 48u) { setLastError("mesh too deep for the traversal stacks"); return HPSDF_ERR_UNSUPPORTED; }
        // meshSampleKernel keeps a wide-node index in bits 0-27 of a stack entry and a group count in bits 28-29
        if (nWide >= (1u << 28)) { setLastError("too many 4-wide BVH nodes for the traversal stack entries"); return HPSDF_ERR_UNSUPPORTED; }
        BvhCountTable counts;
        memset(&counts, 0, sizeof(counts));
        for (const auto& kv : shape.count)
        {
            if (counts.n >= 96) { setLastError("internal: BVH size table overflow"); return HPSDF_ERR_UNSUPPORTED; }
            counts.size[counts.n] = kv.first; counts.count[counts.n] = kv.second; ++counts.n;
        }

        hpsdf_mesh* m = new hpsdf_mesh();
        m->device = ctx->device; m->nTris = nT; m->nVerts = nV;
        auto align = [](size_t x) { return (x + 255) & ~(size_t)255; };
        const size_t bNodes = align((size_t)nNodes * sizeof(BvhNode)), bTv = align((size_t)nT * 48), bPs = align((size_t)nT * 84),
                     bObb = align((size_t)nNodes * 64), bWide = align((size_t)nWide * 128);
        // every block starts on a 256-byte boundary of the blob: each 128-byte wide node is one cache line (mesh_build.cuh: meshWideKernel)
        // the ~200 MB of a large mesh come from the device's cache of released allocations (cudaMalloc + cudaFree of that size
        // cost 5-25 ms, more than the set-up kernels, when meshes are created and destroyed in a loop)
        m->ctx = ctx;
        cudaError_t e = acquireBlob(*ctx, bNodes + bTv + bPs + bObb + bWide + 256, &m->blob, &m->blobBytes);
        if (e != cudaSuccess) { delete m; return failCuda(e, "mesh allocation"); }
        char* p = (char*)m->blob;
        m->view.nodes = (const BvhNode*)p;
        m->view.triVerts = (const void*)(p + bNodes);
        m->view.pseudo = (const float*)(p + bNodes + bTv);
        m->view.nTris = nT; m->view.nNodes = nNodes;
        m->view.obb = (const void*)(p + bNodes + bTv + bPs);
        m->view.wide = (const void*)(p + bNodes + bTv + bPs + bObb);
        m->dView = (DeviceMeshView*)(p + bNodes + bTv + bPs + bObb + bWide);

        std::lock_guard<std::mutex> wsLock(*(std::mutex*)ctx->wsMutex);         // the temporaries live in the device's build workspace
        cudaStream_t stream = ctx->ws.stream;
        auto fail = [&](hpsdf_status st) { cudaStreamSynchronize(stream); releaseBlob(*ctx, m->blob, m->blobBytes); delete m; return st; };
        const size_t bIn = align((size_t)nV * 12) + align((size_t)nT * 12);
        e = ctx->ws.meshTmp.reserve(bIn + meshBuildTempBytes(nT, nNodes));
        if (e != cudaSuccess) return fail(failCuda(e, "mesh workspace"));
        float* dV = (float*)ctx->ws.meshTmp.p;
        uint32_t* dTri = (uint32_t*)(ctx->ws.meshTmp.p + align((size_t)nV * 12));
        const MeshBuildTemp T = carveMeshTemp(ctx->ws.meshTmp.p + bIn, nT, nNodes);
        e = cudaMemcpyAsync(dV, vertices, (size_t)nV * 12, cudaMemcpyHostToDevice, stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(dTri, tri_indices, (size_t)nT * 12, cudaMemcpyHostToDevice, stream);
        if (e != cudaSuccess) return fail(failCuda(e, "mesh upload"));
        stage("upload");
        const MeshBuildIn M{ dV, dTri, nV, nT };

        // half-edge twins (Mesh::CreateHalfEdges, Mesh.cpp:87-131)
        e = meshBuildHalfEdgesAndPseudo(M, T, (float*)m->view.pseudo, stream);
        uint32_t flags[2] = { 0, 0 };
        if (e == cudaSuccess) e = cudaMemcpyAsync(flags, T.flags, 8, cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        if (e != cudaSuccess) return fail(failCuda(e, "mesh half-edges"));
        if (flags[0] & 1u) { setLastError("triangle index out of range"); return fail(HPSDF_ERR_INVALID_ARG); }
        if (flags[0] & 2u) { setLastError("mesh has an edge without a twin: not a closed manifold (Mesh.cpp:121-128)"); return fail(HPSDF_ERR_MESH); }
        stage("half-edges");

        // pseudonormals, BVH levels, refit
        const uint32_t* order = nullptr;
        e = meshBuildBvh(M, T, counts, levels, nNodes, (float*)m->view.pseudo, (BvhNode*)m->view.nodes, &order, stream);
        BvhNode root;
        if (e == cudaSuccess) e = cudaMemcpyAsync(&root, m->view.nodes, sizeof(BvhNode), cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        if (e != cudaSuccess) return fail(failCuda(e, "mesh BVH"));
        memcpy(m->mn, root.mn, 12); memcpy(m->mx, root.mx, 12);                  // CalculateMeshAABB (Mesh.cpp:66-84)
        stage("pseudonormals + bvh");

        // oriented boxes, 4-wide collapse, triangle slots
        double diag2 = 0.0, maxAbs = 0.0;
        for (int d = 0; d < 3; ++d)
        {
            diag2 += ((double)root.mx[d] - root.mn[d]) * ((double)root.mx[d] - root.mn[d]);
            maxAbs = std::max(maxAbs, std::max(std::fabs((double)root.mn[d]), std::fabs((double)root.mx[d])));
        }
        // float32 projection error on the device is ~1e-7 |p|; query points live in a root box of about the mesh's size
        const double inflate = 1e-5 * std::max(std::sqrt(diag2), maxAbs);
        m->view.inflate = (float)inflate;
        e = meshBuildBoxes(M, T, order, nNodes, inflate, m->view.nodes, (float*)m->view.obb, (float*)m->view.wide, (float4*)m->view.triVerts, stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(m->dView, &m->view, sizeof(DeviceMeshView), cudaMemcpyHostToDevice, stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        if (e != cudaSuccess) return fail(failCuda(e, "mesh boxes"));
        stage("boxes + wide + slots");
        *out = m;
        return HPSDF_OK;
    }

    HPSDF_API hpsdf_status hpsdf_mesh_signed_distance(const hpsdf_mesh* mesh, const float* xyz, size_t n, float* out)
    {
        if (!mesh || (n && (!xyz || !out))) { setLastError("null pointer"); return HPSDF_ERR_INVALID_ARG; }
        if (!n) return HPSDF_OK;
        HPSDF_CUDA(cudaSetDevice(mesh->device));
        float *dIn = nullptr, *dOut = nullptr;
        HPSDF_CUDA(cudaMalloc((void**)&dIn, n * 12));
        cudaError_t e = cudaMalloc((void**)&dOut, n * 4);
        if (e == cudaSuccess) e = cudaMemcpy(dIn, xyz, n * 12, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = launchMeshDistance(mesh->dView, dIn, n, dOut, nullptr);
        if (e == cudaSuccess) e = cudaMemcpy(out, dOut, n * 4, cudaMemcpyDeviceToHost);
        cudaFree(dIn); cudaFree(dOut);
        if (e != cudaSuccess) return failCuda(e, "hpsdf_mesh_signed_distance");
        return HPSDF_OK;
    }

    HPSDF_API hpsdf_status hpsdf_mesh_aabb(const hpsdf_mesh* mesh, float mn[3], float mx[3])
    {
        if (!mesh || !mn || !mx) { setLastError("null pointer"); return HPSDF_ERR_INVALID_ARG; }
        memcpy(mn, mesh->mn, 12); memcpy(mx, mesh->mx, 12);
        return HPSDF_OK;
    }

    HPSDF_API void hpsdf_mesh_destroy(hpsdf_mesh* mesh)
    {
        if (!mesh) return;
        cudaSetDevice(mesh->device);
        cudaDeviceSynchronize();                       // what cudaFree did implicitly: nothing in flight may still read the mesh
        if (mesh->ctx) releaseBlob(*mesh->ctx, mesh->blob, mesh->blobBytes);
        else cudaFree(mesh->blob);
        delete mesh;
    }
}
