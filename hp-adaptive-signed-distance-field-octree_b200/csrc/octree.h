// octree.h — host-side objects behind the C ABI: the octree handle (hpsdf_octree), meshes, communicators.
#pragma once
#include <cuda_runtime.h>
#include <mutex>
#include <string>
#include <vector>
#include "hp_common.h"
#include "device_ctx.h"

namespace hpsdf
{
    // thread-local error text behind hpsdf_last_error()
    void setLastError(const std::string& msg);
    hpsdf_status failCuda(cudaError_t e, const char* what);

#define HPSDF_CUDA(call)                                                         \
    do {                                                                         \
        cudaError_t _e = (call);                                                 \
        if (_e != cudaSuccess) return ::hpsdf::failCuda(_e, #call);              \
    } while (0)

    // SDF::Node (Include/HP/Node.h:10-33) on the host, plus the pool slot that holds the leaf's coefficients while building.
    struct HostNode
    {
        uint64_t child  = kNoChild;
        float    mn[3]  = { 0, 0, 0 }, mx[3] = { 0, 0, 0 };
        uint64_t cstart = 0;              // basis.coeffsStart after ReallocCoeffs
        uint32_t slot   = 0;              // build time: offset of the coefficients in the device pool
        uint8_t  degree = kInternalTag;
        uint8_t  depth  = kMaxDepth + 1;
    };
}

struct hpsdf_mesh;

// SDF::Octree (Include/HP/Octree.h:36-176): nodes on the host, coefficients resident on the device.
struct hpsdf_octree
{
    int                 device = 0;
    hpsdf::DeviceCtx*   ctx = nullptr;
    hpsdf_config        cfg{};
    hpsdf::RootMap      map{};
    std::vector<hpsdf::HostNode> nodes;          // host copy of the node array; EMPTY after a device-scheduled Create until something
                                                 // needs it (ensureHostNodes reads the device image back)
    size_t              nNodes = 0;              // node count (authoritative; nodes.size() may be 0)
    size_t              nCoeffs = 0;

    size_t              dBlobBytes = 0;          // capacity of dBlob (it comes from the device's blob cache)
    void*               dBlob = nullptr;         // one allocation: packed store | padded store | QNodes | top table | view
    double*             dCoeffs = nullptr;       // packed store, MemoryBlock order (DFS leaf order)
    double*             dCoeffsPad = nullptr;    // Query layout: every leaf starts at an even index
    size_t              nCoeffsPad = 0;
    hpsdf::QNode*       dNodes = nullptr;
    uint32_t*           dTop = nullptr;          // 16^3 table, or nullptr when the tree is not complete to depth 4
    hpsdf::DeviceTreeView  view{};
    hpsdf::DeviceTreeView* dView = nullptr;      // device copy of `view` (handle of an OCTREE primitive)
    unsigned char*      dNodeImage = nullptr;    // 56-byte SDF::Node records as ToMemoryBlock writes them (valid when imageValid)
    bool                imageValid = false;
    // diagnostics of a device-scheduled build stay on the device until somebody reads them
    size_t              nLogDev = 0;             // apply-log entries in dApplyLog (fetched by ensureApplyLog)
    hpsdf_apply_log_entry* dApplyLog = nullptr;
    double*             dLeafErr = nullptr;      // current error per node at termination (input of the cut-tie log)
    bool                logOnDevice = false;

    hpsdf_build_stats   stats{};
    std::vector<hpsdf_decision_log_entry> decisionLog;
    std::vector<hpsdf_apply_log_entry>    applyLog;
    // inputs of the cut-tie log of a device-scheduled build; the group is worked out when the decision log is first read
    size_t              cutLogStart = 0;
    double              cutTotalBeforeLast = 0.0, cutCheck = 0.0;
    bool                cutLogPending = false, cutQueueEmpty = false;

    // scratch of the host-pointer Query path
    std::mutex          queryMutex;
    double*             dScratchIn[3]  = { nullptr, nullptr, nullptr };
    double*             dScratchOut[3] = { nullptr, nullptr, nullptr };
    size_t              scratchPts = 0;
    cudaStream_t        qStreams[3] = { nullptr, nullptr, nullptr };

    ~hpsdf_octree();
};

namespace hpsdf
{
    void          setRootMap(const hpsdf_config& cfg, RootMap& map);
    // One device allocation for everything a finished tree owns; sized by t.nNodes, t.nCoeffs and t.nCoeffsPad.
    hpsdf_status  allocTreeBlob(hpsdf_octree& t);
    // t.nCoeffsPad from the host nodes (every leaf starts at an even index of the Query store)
    size_t        paddedCoeffCount(const hpsdf_octree& t);
    // Host copy of the node array, read back from the device image if the build left it on the device.
    hpsdf_status  ensureHostNodes(hpsdf_octree& t);
    // Completes the decision log of a device-scheduled build (the equal-error group at the termination cut).
    void          ensureDecisionLog(hpsdf_octree& t);
    // Fetches the apply log of a device-scheduled build.
    void          ensureApplyLog(hpsdf_octree& t);
    // Build QNodes, the padded coefficient store and the top table from nodes + dCoeffs.
    hpsdf_status  finalizeQueryStructures(hpsdf_octree& t, cudaStream_t stream);
    // Fill t.view from the tree's device arrays (top: the depth-4 table, or nullptr) and copy it to t.dView on `stream`.
    cudaError_t   uploadTreeView(hpsdf_octree& t, const uint32_t* top, cudaStream_t stream);
    // SDF program with handles resolved to device views; fails on malformed programs.
    hpsdf_status  resolveProgram(const hpsdf_sdf_program* prog, int device, SdfProgramDev& out);
    // Octree::Create on the device (build.cpp)
    hpsdf_status  buildOctree(hpsdf_octree& t, const hpsdf_build_opts& opts, const SdfProgramDev& prog);
    // PerformContinuityPostProcess on the device (continuity.cpp + kernels)
    hpsdf_status  continuityPostProcess(hpsdf_octree& t, const hpsdf_build_opts& opts, cudaStream_t stream);
    hpsdf_status  toMemoryBlock(const hpsdf_octree& t, size_t* size, void** ptr);
    hpsdf_status  fromMemoryBlock(hpsdf_octree& t, const void* ptr, size_t size);
    hpsdf_status  queryHost(hpsdf_octree& t, const double* xyz, size_t n, double* out);
    const std::string& lastError();
    const DeviceMeshView* meshDeviceView(const hpsdf_mesh* m);      // mesh.cpp
    int           meshDevice(const hpsdf_mesh* m);
    // CornerAABB (Octree.cpp:1096-1112)
    void          cornerAabb(const HostNode& parent, uint32_t i, float mn[3], float mx[3]);
    double        nowMs();
}
