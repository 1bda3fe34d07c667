// build_common.h — what both schedulers of Octree::Create share (build.cpp: host replay, build_device.cpp: device-resident).
#pragma once
#include <vector>
#include "octree.h"

namespace hpsdf
{
    // ReallocCoeffs (Octree.cpp:474-555): DFS from the root's children by child slot; leaves packed in visiting order into
    // t.dCoeffs from their pool slots (t.nodes[i].slot); sets cstart of every leaf and t.nCoeffs, allocates the tree blob.
    hpsdf_status packCoefficients(hpsdf_octree& t, const double* pool, cudaStream_t stream);

    // Near-threshold divergence log (BASELINE north_star): the greedy loop stops in the middle of a run of leaves whose
    // errors are equal to rounding (mirror-symmetric cells have errors equal to the last bits). WHICH of them were
    // refined before the cut depends on the last bits, so another implementation of the same algorithm may refine
    // other members of the group. Logs the whole group: kind 2 = refined before the cut, kind 3 = left unrefined.
    // errOf: current error per node; levelLogStart: first apply-log entry of the last batch of applied jobs.
    void logCutTieGroup(hpsdf_octree& t, const std::vector<double>& errOf, size_t levelLogStart, bool queueEmpty);

    // The fit launches of one round, for both schedulers (ps = summarizeProgram(prog), worked out once per build): cnt[d]
    // fits of degree d at the task positions and pool slots of `lay`, already expanded into t.ctx->ws.tasks
    // (launchExpandJobsDev) with the pool reserved. One kernel per degree present (this rank's shard), highest degree first,
    // fanned out over the workspace's four auxiliary streams; evBegin / evEnd bracket the launches on `stream`. A sharded
    // round ends with one grouped broadcast per (degree group, rank).
    hpsdf_status launchRoundFits(hpsdf_octree& t, const hpsdf_build_opts& o, const SdfProgramDev& prog, const ProgramSummary& ps,
                                 cudaStream_t stream, const uint32_t* cnt, const RoundLayout& lay, uint32_t nTasks, int rank, int world,
                                 cudaEvent_t evBegin, cudaEvent_t evEnd);

    hpsdf_status buildOctreeHost(hpsdf_octree& t, const hpsdf_build_opts& opts, const SdfProgramDev& prog);
    hpsdf_status buildOctreeDevice(hpsdf_octree& t, const hpsdf_build_opts& opts, const SdfProgramDev& prog, bool& fallBack);
}
