// tree.cpp — the finished octree: Query structures, MemoryBlock I/O, SDF-program resolution.
//
// Reference: ToMemoryBlock / FromMemoryBlock (Source/HP/Octree.cpp:424-456 / 403-421), LP64 byte layout (SURVEY.md App. B):
//   [u64 nCoeffs][f64 x nCoeffs][u64 nNodes][Node x nNodes, 56 B each][Config, 80 B]
//   Node: childIdx u64 @0 | aabb.min 3xf32 @8 | aabb.max 3xf32 @20 | coeffsStart u64 @32 | degree u8 @40 | depth u8 @48.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include "octree.h"

hpsdf_octree::~hpsdf_octree()
{
    if (ctx) { cudaSetDevice(device); hpsdf::releaseBlob(*ctx, dBlob, dBlobBytes); }
    else cudaFree(dBlob);
    for (int i = 0; i < 3; ++i)
    {
        cudaFree(dScratchIn[i]); cudaFree(dScratchOut[i]);
        if (qStreams[i]) cudaStreamDestroy(qStreams[i]);
    }
}

namespace hpsdf
{
    size_t paddedCoeffCount(const hpsdf_octree& t)
    {
        size_t pad = 0;
        for (const HostNode& n : t.nodes) if (n.child == kNoChild) pad += ((size_t)coeffCount(n.degree) + 1u) & ~(size_t)1u;
        return pad;
    }

    hpsdf_status allocTreeBlob(hpsdf_octree& t)
    {
        auto align = [](size_t b) { return (b + 255) & ~(size_t)255; };
        const size_t nNodes = t.nNodes;
        const size_t bCoeffs = align(std::max<size_t>(t.nCoeffs, 1) * 8), bPad = align(std::max<size_t>(t.nCoeffsPad, 2) * 8);
        const size_t bNodes = align(nNodes * sizeof(QNode)), bTop = align(4096 * 4), bView = align(sizeof(DeviceTreeView)), bImage = align(nNodes * 56);
        const size_t bLog = align(t.nLogDev * sizeof(hpsdf_apply_log_entry)), bErr = t.nLogDev ? align(nNodes * 8) : 0;
        const size_t need = bCoeffs + bPad + bNodes + bTop + bView + bImage + bLog + bErr;
        if (!t.dBlob || t.dBlobBytes < need || t.dBlobBytes > 4 * need + ((size_t)1 << 20))
        {
            releaseBlob(*t.ctx, t.dBlob, t.dBlobBytes);
            t.dBlob = nullptr; t.dBlobBytes = 0;
            HPSDF_CUDA(acquireBlob(*t.ctx, need, &t.dBlob, &t.dBlobBytes));
        }
        char* p = (char*)t.dBlob;
        t.dCoeffs = (double*)p; p += bCoeffs;
        t.dCoeffsPad = (double*)p; p += bPad;
        t.dNodes = (QNode*)p; p += bNodes;
        t.dTop = (uint32_t*)p; p += bTop;
        t.dView = (DeviceTreeView*)p; p += bView;
        t.dNodeImage = (unsigned char*)p; p += bImage;
        t.dApplyLog = (hpsdf_apply_log_entry*)p; p += bLog;
        t.dLeafErr = (double*)p;
        t.imageValid = false; t.logOnDevice = false;
        return HPSDF_OK;
    }

    hpsdf_status finalizeQueryStructures(hpsdf_octree& t, cudaStream_t stream)
    {
        const size_t nNodes = t.nodes.size();
        if (nNodes != t.nNodes) { setLastError("internal: host node array does not match the tree"); return HPSDF_ERR_CUDA; }
        if (nNodes >= 0xFFFFFFFFull) { setLastError("too many nodes for the 32-bit query layout"); return HPSDF_ERR_UNSUPPORTED; }
        // staging: [QNodes][top 4096][src|dst|count segments] in one pinned buffer, one H2D copy
        size_t nLeaves = 0;
        for (const HostNode& n : t.nodes) nLeaves += n.child == kNoChild;
        const size_t wNodes = nNodes * 4, wTop = 4096, wSeg = 3 * nLeaves;
        BuildWorkspace& ws = t.ctx->ws;
        HPSDF_CUDA(ws.hSegs.reserve(wNodes + wTop + wSeg + 16));
        HPSDF_CUDA(ws.segs.reserve(wSeg + 16));
        QNode* q = (QNode*)ws.hSegs.p;
        uint32_t* top = ws.hSegs.p + wNodes;
        uint32_t* srcOff = top + wTop; uint32_t* dstOff = srcOff + nLeaves; uint32_t* count = dstOff + nLeaves;
        size_t padCur = 0, li = 0;
        for (size_t i = 0; i < nNodes; ++i)
        {
            const HostNode& n = t.nodes[i];
            q[i].depth = n.depth;
            if (n.child == kNoChild)
            {
                const uint32_t c = (uint32_t)coeffCount(n.degree);
                q[i].child = 0xFFFFFFFFu; q[i].degree = n.degree; q[i].cstart = (uint32_t)padCur;
                srcOff[li] = (uint32_t)n.cstart; dstOff[li] = (uint32_t)padCur; count[li] = c; ++li;
                padCur += (c + 1u) & ~1u;                                // next leaf starts at an even index (16-byte aligned)
            }
            else { q[i].child = (uint32_t)n.child; q[i].degree = kInternalTag; q[i].cstart = 0; }
        }
        if (padCur >= 0xFFFFFFF0ull) { setLastError("coefficient store exceeds the 32-bit query layout"); return HPSDF_ERR_UNSUPPORTED; }

        // depth-4 entry table: valid only if every 16^3 cell exists at depth 4 (always true for trees the reference builds)
        bool topOk = true;
        for (uint32_t code = 0; code < 4096 && topOk; ++code)
        {
            const uint32_t ix = code & 15, iy = (code >> 4) & 15, iz = code >> 8;
            uint64_t cur = 0;
            for (int l = 3; l >= 0; --l)
            {
                if (t.nodes[cur].child == kNoChild) { topOk = false; break; }
                cur = t.nodes[cur].child + ((ix >> l) & 1) + 2 * ((iy >> l) & 1) + 4 * ((iz >> l) & 1);
            }
            top[code] = (uint32_t)cur;
        }
        if (padCur != t.nCoeffsPad || !t.dBlob) { setLastError("internal: tree blob not allocated for this tree"); return HPSDF_ERR_CUDA; }

        HPSDF_CUDA(cudaMemcpyAsync(t.dNodes, q, nNodes * sizeof(QNode), cudaMemcpyHostToDevice, stream));
        HPSDF_CUDA(cudaMemcpyAsync(t.dTop, top, 4096 * 4, cudaMemcpyHostToDevice, stream));
        HPSDF_CUDA(cudaMemcpyAsync(ws.segs.p, srcOff, wSeg * 4, cudaMemcpyHostToDevice, stream));
        HPSDF_CUDA(cudaMemsetAsync(t.dCoeffsPad, 0, std::max<size_t>(padCur, 2) * 8, stream));
        HPSDF_CUDA(launchGatherSegments(t.dCoeffs, t.dCoeffsPad, ws.segs.p, ws.segs.p + nLeaves, ws.segs.p + 2 * nLeaves, (uint32_t)nLeaves, stream));
        t.stats.kernel_launches++;
        HPSDF_CUDA(uploadTreeView(t, topOk ? t.dTop : nullptr, stream));
        HPSDF_CUDA(cudaStreamSynchronize(stream));
        return HPSDF_OK;
    }

    cudaError_t uploadTreeView(hpsdf_octree& t, const uint32_t* top, cudaStream_t stream)
    {
        t.view.nodes = t.dNodes; t.view.coeffs = t.dCoeffsPad; t.view.top = top; t.view.bidx = t.ctx->fitTab.bidx;
        t.view.map = t.map; t.view.nNodes = (uint32_t)t.nNodes;
        return cudaMemcpyAsync(t.dView, &t.view, sizeof(DeviceTreeView), cudaMemcpyHostToDevice, stream);
    }

    hpsdf_status resolveProgram(const hpsdf_sdf_program* prog, int device, SdfProgramDev& out)
    {
        if (!prog || !prog->instr || prog->n_instr == 0 || prog->n_instr > HPSDF_PROGRAM_MAX_INSTR)
        {
            setLastError("SDF program is null, empty or longer than HPSDF_PROGRAM_MAX_INSTR");
            return HPSDF_ERR_INVALID_ARG;
        }
        memset(&out, 0, sizeof(out));
        out.n = prog->n_instr;
        int sp = 0;
        for (uint32_t i = 0; i < prog->n_instr; ++i)
        {
            const hpsdf_sdf_instr& in = prog->instr[i];
            SdfInstrDev& o = out.instr[i];
            o.op = in.op;
            memcpy(o.p, in.p, sizeof(o.p));
            switch (in.op)
            {
                case HPSDF_PRIM_TORUS:
                {
                    const int axis = (int)in.p[5];
                    if (axis < 0 || axis > 2 || (double)axis != in.p[5]) { setLastError("TORUS axis must be 0, 1 or 2"); return HPSDF_ERR_INVALID_ARG; }
                    o.op = axis == 0 ? kOpTorusX : axis == 1 ? kOpTorusY : kOpTorusZ;
                    ++sp; break;
                }
                case HPSDF_PRIM_SPHERE: case HPSDF_PRIM_BOX: case HPSDF_PRIM_CAPSULE: case HPSDF_PRIM_PLANE:
                    ++sp; break;
                case HPSDF_PRIM_OCTREE:
                {
                    const hpsdf_octree* src = (const hpsdf_octree*)in.handle;
                    if (!src || !src->dView || src->device != device) { setLastError("OCTREE primitive needs a finished tree on the same device"); return HPSDF_ERR_INVALID_ARG; }
                    o.handle = src->dView; ++sp; break;
                }
                case HPSDF_PRIM_MESH:
                {
                    const hpsdf_mesh* src = (const hpsdf_mesh*)in.handle;
                    if (!src || meshDevice(src) != device) { setLastError("MESH primitive needs a mesh created on the same device"); return HPSDF_ERR_INVALID_ARG; }
                    o.handle = meshDeviceView(src); ++sp; break;
                }
                case HPSDF_OP_NEGATE:
                    if (sp < 1) { setLastError("SDF program: operator without operand"); return HPSDF_ERR_INVALID_ARG; }
                    break;
                case HPSDF_OP_UNION: case HPSDF_OP_INTERSECT: case HPSDF_OP_SUBTRACT:
                    if (sp < 2) { setLastError("SDF program: binary operator needs two operands"); return HPSDF_ERR_INVALID_ARG; }
                    --sp; break;
                default:
                    setLastError("SDF program: unknown opcode");
                    return HPSDF_ERR_INVALID_ARG;
            }
            if (sp > HPSDF_PROGRAM_MAX_STACK) { setLastError("SDF program: stack deeper than HPSDF_PROGRAM_MAX_STACK"); return HPSDF_ERR_INVALID_ARG; }
        }
        if (sp != 1) { setLastError("SDF program must leave exactly one value"); return HPSDF_ERR_INVALID_ARG; }
        return HPSDF_OK;
    }

    // ToMemoryBlock (Octree.cpp:424-456)
    hpsdf_status toMemoryBlock(const hpsdf_octree& t, size_t* size, void** ptr)
    {
        const size_t nC = t.nCoeffs, nN = t.nNodes;
        const size_t bytes = 8 + 8 * nC + 8 + 56 * nN + 80;
        uint8_t* p = (uint8_t*)malloc(bytes);                     // malloc-owned, the caller free()s it (Octree.cpp:445)
        if (!p) { setLastError("malloc failed"); return HPSDF_ERR_OOM; }
        const uint64_t nc = nC, nn = nN;                           // (every byte is written below: no memset of the 8 nC payload)
        memcpy(p, &nc, 8);
        if (nC)
        {
            cudaSetDevice(t.device);
            cudaError_t e = cudaMemcpy(p + 8, t.dCoeffs, 8 * nC, cudaMemcpyDeviceToHost);
            if (e != cudaSuccess) { free(p); return failCuda(e, "ToMemoryBlock copy"); }
        }
        uint8_t* q = p + 8 + 8 * nC;
        memcpy(q, &nn, 8); q += 8;
        if (t.nodes.empty() && t.imageValid)
        {
            // the build left the SDF::Node records on the device (finish_kernels.cuh: emitTreeKernel): one more copy
            cudaError_t e = cudaMemcpy(q, t.dNodeImage, 56 * nN, cudaMemcpyDeviceToHost);
            if (e != cudaSuccess) { free(p); return failCuda(e, "ToMemoryBlock copy"); }
            q += 56 * nN;
        }
        else for (size_t i = 0; i < nN; ++i, q += 56)
        {
            const HostNode& n = t.nodes[i];
            memcpy(q, &n.child, 8); memcpy(q + 8, n.mn, 12); memcpy(q + 20, n.mx, 12);
            const uint64_t deg = n.degree, dep = n.depth;            // u8 + 7 bytes of zero padding each (LP64 layout of SDF::Node)
            memcpy(q + 32, &n.cstart, 8); memcpy(q + 40, &deg, 8); memcpy(q + 48, &dep, 8);
        }
        memcpy(q, &t.cfg, 80);
        *size = bytes; *ptr = p;
        return HPSDF_OK;
    }

    // FromMemoryBlock (Octree.cpp:403-421); validates what the reference only asserts.
    hpsdf_status fromMemoryBlock(hpsdf_octree& t, const void* ptr, size_t size)
    {
        const uint8_t* p = (const uint8_t*)ptr;
        if (!p || size < 96) { setLastError("MemoryBlock is null or too small"); return HPSDF_ERR_BAD_BLOCK; }
        uint64_t nc = 0, nn = 0;
        memcpy(&nc, p, 8);
        if (nc > (size - 96) / 8) { setLastError("MemoryBlock: coefficient count exceeds the block"); return HPSDF_ERR_BAD_BLOCK; }
        memcpy(&nn, p + 8 + 8 * nc, 8);
        if (nn == 0 || nn > (size - 96 - 8 * nc) / 56 || size != 8 + 8 * nc + 8 + 56 * nn + 80)
        {
            setLastError("MemoryBlock: size does not match 96 + 8 nCoeffs + 56 nNodes");
            return HPSDF_ERR_BAD_BLOCK;
        }
        memcpy(&t.cfg, p + 16 + 8 * nc + 56 * nn, 80);
        setRootMap(t.cfg, t.map);
        t.nodes.resize(nn);
        const uint8_t* q = p + 16 + 8 * nc;
        for (uint64_t i = 0; i < nn; ++i, q += 56)
        {
            HostNode& n = t.nodes[i];
            memcpy(&n.child, q, 8); memcpy(n.mn, q + 8, 12); memcpy(n.mx, q + 20, 12);
            memcpy(&n.cstart, q + 32, 8); n.degree = q[40]; n.depth = q[48];
        }
        // structural checks: links in range, leaves inside the store, dyadic cells (the Query kernel tracks cell centres
        // instead of loading AABBs, which is exact only for the reference's CornerAABB layout)
        for (int a = 0; a < 3; ++a)
            if (t.nodes[0].mn[a] != -0.5f || t.nodes[0].mx[a] != 0.5f) { setLastError("MemoryBlock: root is not [-0.5,0.5]^3"); return HPSDF_ERR_BAD_BLOCK; }
        if (t.nodes[0].child == kNoChild) { setLastError("MemoryBlock: root has no children"); return HPSDF_ERR_BAD_BLOCK; }
        for (uint64_t i = 0; i < nn; ++i)
        {
            const HostNode& n = t.nodes[i];
            if (n.child == kNoChild)
            {
                if (n.degree > kMaxDegree || n.depth > kMaxDepth || n.cstart + (uint64_t)coeffCount(n.degree) > nc)
                { setLastError("MemoryBlock: leaf outside the coefficient store"); return HPSDF_ERR_BAD_BLOCK; }
            }
            else
            {
                if (n.child >= nn || nn - n.child < 8 || n.child <= i) { setLastError("MemoryBlock: child index out of range"); return HPSDF_ERR_BAD_BLOCK; }
                for (uint32_t c = 0; c < 8; ++c)
                {
                    float mn[3], mx[3];
                    cornerAabb(n, c, mn, mx);
                    const HostNode& ch = t.nodes[n.child + c];
                    if (memcmp(mn, ch.mn, 12) || memcmp(mx, ch.mx, 12) || ch.depth != n.depth + 1)
                    { setLastError("MemoryBlock: node boxes are not the reference's CornerAABB layout"); return HPSDF_ERR_BAD_BLOCK; }
                }
            }
        }
        t.nCoeffs = nc; t.nNodes = nn; t.nCoeffsPad = paddedCoeffCount(t);
        hpsdf_status st = allocTreeBlob(t);
        if (st != HPSDF_OK) return st;
        HPSDF_CUDA(cudaMemcpy(t.dCoeffs, p + 8, nc * 8, cudaMemcpyHostToDevice));
        uint64_t leaves = 0;
        for (const HostNode& n : t.nodes) leaves += n.child == kNoChild;
        t.stats.n_nodes = nn; t.stats.n_leaves = leaves; t.stats.n_coeffs = nc;
        std::lock_guard<std::mutex> wsLock(*(std::mutex*)t.ctx->wsMutex);
        return finalizeQueryStructures(t, t.ctx->ws.stream);
    }

    hpsdf_status ensureHostNodes(hpsdf_octree& t)
    {
        if (!t.nodes.empty() || t.nNodes == 0) return HPSDF_OK;
        if (!t.imageValid) { setLastError("internal: tree has neither host nodes nor a device image"); return HPSDF_ERR_CUDA; }
        std::vector<uint8_t> img(56 * t.nNodes);
        HPSDF_CUDA(cudaSetDevice(t.device));
        HPSDF_CUDA(cudaMemcpy(img.data(), t.dNodeImage, img.size(), cudaMemcpyDeviceToHost));
        t.nodes.resize(t.nNodes);
        const uint8_t* q = img.data();
        for (size_t i = 0; i < t.nNodes; ++i, q += 56)
        {
            HostNode& n = t.nodes[i];
            memcpy(&n.child, q, 8); memcpy(n.mn, q + 8, 12); memcpy(n.mx, q + 20, 12);
            memcpy(&n.cstart, q + 32, 8); n.degree = q[40]; n.depth = q[48];
        }
        return HPSDF_OK;
    }

    // Octree::Query for host arrays: chunks of points go H2D -> kernel -> D2H on three rotating streams so the copies of
    // one chunk overlap the kernel of another (PCIe is full duplex).
    hpsdf_status queryHost(hpsdf_octree& t, const double* xyz, size_t n, double* out)
    {
        if (!n) return HPSDF_OK;
        std::lock_guard<std::mutex> lock(t.queryMutex);
        HPSDF_CUDA(cudaSetDevice(t.device));
        // at least 8 chunks for a large call, so the H2D copy of one chunk overlaps the kernel and the D2H copy of the previous
        // ones (a single 2^22-point chunk serialised the three: 1.55e9 points/s where the H2D engine alone allows 2.2e9)
        const size_t chunk = std::min<size_t>(std::max<size_t>((n + 7) / 8, (size_t)1 << 16), (size_t)1 << 22);
        if (t.scratchPts < chunk)
        {
            for (int i = 0; i < 3; ++i)
            {
                cudaFree(t.dScratchIn[i]); cudaFree(t.dScratchOut[i]);
                t.dScratchIn[i] = t.dScratchOut[i] = nullptr;
                HPSDF_CUDA(cudaMalloc((void**)&t.dScratchIn[i], chunk * 24));
                HPSDF_CUDA(cudaMalloc((void**)&t.dScratchOut[i], chunk * 8));
                if (!t.qStreams[i]) HPSDF_CUDA(cudaStreamCreateWithFlags(&t.qStreams[i], cudaStreamNonBlocking));
            }
            t.scratchPts = chunk;
        }
        int s = 0;
        for (size_t off = 0; off < n; off += chunk, s = (s + 1) % 3)
        {
            const size_t m = std::min(chunk, n - off);
            HPSDF_CUDA(cudaMemcpyAsync(t.dScratchIn[s], xyz + 3 * off, m * 24, cudaMemcpyHostToDevice, t.qStreams[s]));
            HPSDF_CUDA(launchQuery(t.view, t.dScratchIn[s], m, t.dScratchOut[s], t.ctx->smCount, t.qStreams[s]));
            HPSDF_CUDA(cudaMemcpyAsync(out + off, t.dScratchOut[s], m * 8, cudaMemcpyDeviceToHost, t.qStreams[s]));
        }
        for (int i = 0; i < 3; ++i) HPSDF_CUDA(cudaStreamSynchronize(t.qStreams[i]));
        return HPSDF_OK;
    }
}
