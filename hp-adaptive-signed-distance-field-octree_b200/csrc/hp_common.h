// hp_common.h — constants, tables and plain structs shared by the host scheduler and the CUDA kernels.
//
// Reference constants: Include/HP/Consts.h:7-8 (BASIS_MAX_DEGREE = 12, TREE_MAX_DEPTH = 10), Include/HP/Utility.h:40-196
// (SumToN, NormalisedLengths, LegendreCoeffientCount, LegendreCoefficent, BasisIndexValues, SharedFaceLookup).
// The tables are rebuilt here from their definitions; nothing is copied from the reference.
#pragma once
#ifdef __CUDACC_RTC__
// run-time compilation (NVRTC, jit.cpp): no system headers
typedef unsigned char uint8_t; typedef unsigned short uint16_t; typedef unsigned int uint32_t; typedef unsigned long long uint64_t;
typedef int int32_t; typedef long long int64_t; typedef unsigned long size_t;
#define HPSDF_NO_SYSTEM_HEADERS 1
#else
#include <cstdint>
#include <cstddef>
#endif
#include "../../include/hpsdf.h"

#if defined(__CUDACC__)
#define HPSDF_HD __host__ __device__
#else
#define HPSDF_HD
#endif

namespace hpsdf
{
    constexpr int      kMaxDegree   = 12;                    // BASIS_MAX_DEGREE
    constexpr int      kMaxDepth    = 10;                    // TREE_MAX_DEPTH
    constexpr uint8_t  kInternalTag = 13;                    // BASIS_MAX_DEGREE + 1 (Node.cpp:12): degree tag of internal nodes
    constexpr uint64_t kNoChild     = 0xFFFFFFFFFFFFFFFFull; // childIdx = -1 (Node.cpp:8)
    constexpr double   kInitialErr  = 100.0;                 // INITIAL_NODE_ERR (Octree.h:89)
    constexpr int      kCoarseDepth = 4, kCoarseDegree = 2;  // UniformlyRefine (Octree.cpp:115-116)
    constexpr int      kMaxCoeffs   = 455;
    // internal opcodes: HPSDF_PRIM_TORUS with its axis parameter resolved when the program is uploaded
    constexpr uint32_t kOpTorusX = 48, kOpTorusY = 49, kOpTorusZ = 50;

    // LegendreCoeffientCount (Utility.h:87-106). The reference evaluates (u32)((1.0/6.0)*(i+1)*(i+2)*(i+3)) in f64, which
    // truncates to 83 (not 84) at i = 6. The value is part of the MemoryBlock contract (a degree-6 leaf stores 83
    // coefficients; a 6->7 p-fit recomputes index 83 = (6,0,0) with the degree-7 rule), so it is reproduced, not fixed.
    HPSDF_HD constexpr int coeffCount(int degree)
    {
        return degree == 6 ? 83 : (degree + 1) * (degree + 2) * (degree + 3) / 6;
    }
    // number of (b, c) pairs with b + c <= d
    HPSDF_HD constexpr int pairCount(int d) { return (d + 1) * (d + 2) / 2; }
    // User-space coordinate of a Gauss-Legendre node: node -> cell (Octree.cpp:1039) -> root box (Octree.cpp:327). One
    // definition, so the fit kernels and the sample kernel contract it identically.
    HPSDF_HD inline double samplePos(double root, double half, double c, double size, double centre) { return (root * half + c) * size + centre; }
    // Gauss-Legendre points per axis of a degree-d fit (Octree.cpp:1016-1017: rule 4d+1)
    HPSDF_HD constexpr int fitRule(int d) { return 4 * d + 1; }
    // fit kernel geometry (fit_kernel_body.cuh): fits per CTA, threads per CTA and dynamic shared memory per degree.
    // A fit has n^2 columns of samples, one thread each: 25 / 81 / 169 for d = 1..3 would leave 22 / 16 / 12 % of the lanes
    // of a CTA idle, so those degrees pack several fits into one CTA (125 of 128, 243 of 256, 507 of 512 lanes busy).
    // Two degree-4 fits in a 608-thread CTA measured 15 % slower than one in 320 (occupancy).
    HPSDF_HD constexpr int fitGroup(int d)   { return d == 1 ? 5 : (d == 2 || d == 3) ? 3 : 1; }
    HPSDF_HD constexpr int fitPasses(int d)  { return (fitGroup(d) * fitRule(d) * fitRule(d) + 639) / 640; }
    HPSDF_HD constexpr int fitThreads(int d)
    {
        return (((fitGroup(d) * fitRule(d) * fitRule(d) + fitPasses(d) - 1) / fitPasses(d)) + 31) / 32 * 32;
    }
    // shared memory (doubles): Q (d+1)*n | roots n | then per fit of the group: user-space z n | T1 (d+1)*n*n | T2 pairCount*n ;
    // coefficients alias T1
    HPSDF_HD constexpr size_t fitSmemPerFit(int d)
    {
        return (size_t)fitRule(d) + (size_t)(d + 1) * fitRule(d) * fitRule(d) + (size_t)pairCount(d) * fitRule(d);
    }
    HPSDF_HD constexpr size_t fitSmemDoubles(int d)
    {
        return (size_t)(d + 1) * fitRule(d) + fitRule(d) + (size_t)fitGroup(d) * fitSmemPerFit(d);
    }
#ifndef __CUDACC_RTC__
    // Sum-factorised FLOPs of one full fit at degree d, SDF evaluation excluded (SURVEY.md §8d):
    // 2(d+1)n^3 + 2 T2(d) n^2 + 2 N_d n + 4 n^3.
    inline double fitFlops(int d)
    {
        const double n = fitRule(d);
        return 2.0 * (d + 1) * n * n * n + 2.0 * pairCount(d) * n * n + 2.0 * ((d + 1) * (d + 2) * (d + 3) / 6) * n + 4.0 * n * n * n;
    }

    // FLOPs of one evaluation of a primitive / operator, counting sqrt and divide as one each (they expand to ~25-30 FP64
    // instructions on the device): the c_F term of the SURVEY.md §8d formula. 6 more for the unit-cube -> root map.
    inline double sdfOpFlops(uint32_t op)
    {
        switch (op)
        {
            case HPSDF_PRIM_SPHERE:  return 10.0;   // 3 sub, 3 mul, 2 add, sqrt, sub
            case HPSDF_PRIM_BOX:     return 22.0;   // 3 sub, 3 abs, 3 sub, 3 max, 3 mul, 2 add, sqrt, 2 max, min, add
            case HPSDF_PRIM_TORUS: case kOpTorusX: case kOpTorusY: case kOpTorusZ: return 13.0;   // 3 sub, 2 mul, add, sqrt, sub, 2 mul, add, sqrt, sub
            case HPSDF_PRIM_CAPSULE: return 32.0;   // 6 sub, 2 dot (5 each), div, 2 clamp, 3 fma (6), 5, sqrt, sub
            case HPSDF_PRIM_PLANE:   return 6.0;
            case HPSDF_OP_NEGATE:    return 1.0;
            case HPSDF_OP_UNION: case HPSDF_OP_INTERSECT: return 1.0;
            case HPSDF_OP_SUBTRACT:  return 2.0;
            default:                 return 0.0;    // mesh / octree primitives: report evaluations per second instead
        }
    }

    // Host-side tables (tables.cpp)
    struct Tables
    {
        double  nl[kMaxDegree + 1][kMaxDepth + 1];   // NormalisedLengths[a][depth] = sqrt((2a+1) 2^depth), Newton-iterated as Utility.h:25-35
        double  rec[kMaxDegree + 1][2];              // (2i-1)/i, (i-1)/i
        uint8_t bidx[kMaxCoeffs][3];                 // BasisIndexValues: shell p, then i, then j; k = p-i-j
        uint8_t face[3][4][2];                       // SharedFaceLookup[dim][j] = (low child, high child)
    };
    const Tables& tables();
    // Gauss-Legendre rule with n points (1..64), nodes ascending: pointers to n roots / n weights
    const double* glRoots(int n);
    const double* glWeights(int n);
#endif   // !__CUDACC_RTC__

    // ---- device-side descriptors ------------------------------------------------------------------------------
    // Unit cube -> user space map of Octree::Create (Octree.cpp:322-328) and its f32-rounded inverse used by Query
    // (Octree.cpp:323, 420, 665).
    struct RootMap
    {
        double centre[3];
        double sizes[3];
        double invSizes[3];     // (double)(1.0f / size_f32)
    };

    // One FitPolynomial call (Octree.cpp:1007-1093) of a round. 32 bytes.
    struct FitTask
    {
        float    cx, cy, cz, half;   // cell centre and half size in the internal unit cube (dyadic: exact in f32)
        uint32_t out;                // offset (in doubles) of the output coefficient slot in the pool
        uint32_t src;                // offset of the slot whose lower shells are kept (p-fit), or kNoSrc (from scratch)
        uint8_t  depth;              // tree depth of the cell (selects NormalisedLengths[.][depth])
        uint8_t  degree;             // target degree d
        uint8_t  degreeIn;           // degree of the kept lower shells (0 = from scratch)
        uint8_t  pad;
        uint32_t rec;                // index of the result record
    };
    constexpr uint32_t kNoSrc = 0xFFFFFFFFu;

    // One refinement job of a round as a scheduler writes it (32 bytes instead of 9 FitTasks): expandJobsDevKernel turns it
    // into the 8 child fits @degree at task positions hPos..hPos+7 of that degree's group and the p-fit @degree+1 at pPos.
    struct JobDesc
    {
        float    cx, cy, cz, half;   // the parent cell
        uint32_t hPos, pPos;         // task (= record) index of child 0 / of the p-fit
        uint32_t src;                // pool slot of the parent's coefficients (kept shells of the p-fit)
        uint8_t  depth, degree;      // of the parent
        uint8_t  flags;              // 1 = child fits wanted, 2 = p-fit wanted, 4 = coarse cell (one from-scratch fit @kCoarseDegree at pPos)
        uint8_t  pad;
    };
    // where each degree's tasks and output slots start in this round
    struct RoundLayout
    {
        uint32_t groupBegin[kMaxDegree + 2];
        uint32_t groupPool[kMaxDegree + 2];
    };

    // The layout of a round with cnt[d] fits of degree d (d = 1..kMaxDegree): tasks in degree order, output slots handed out
    // in task order from pool offset poolUsed, so a degree group (and a rank's shard of it) is one contiguous range of tasks
    // and one of the pool. Returns the number of tasks; poolEnd = the pool offset after the round (callers refuse a round
    // that takes it past 2^32 doubles).
    HPSDF_HD inline uint32_t layoutRound(const uint32_t* cnt, uint32_t poolUsed, uint32_t* groupBegin, uint32_t* groupPool, uint64_t& poolEnd)
    {
        uint32_t nTasks = 0;
        uint64_t pool = poolUsed;
        groupBegin[0] = 0; groupPool[0] = poolUsed;
        for (int d = 1; d <= kMaxDegree; ++d)
        {
            groupBegin[d] = nTasks; groupPool[d] = (uint32_t)pool;
            nTasks += cnt[d]; pool += (uint64_t)cnt[d] * (uint64_t)coeffCount(d);
        }
        groupBegin[kMaxDegree + 1] = nTasks; groupPool[kMaxDegree + 1] = (uint32_t)pool;
        poolEnd = pool;
        return nTasks;
    }

    // Several GPUs evaluate contiguous shards of each degree group of a round, and selection order is spatially coherent (far
    // and near cells of a mesh cluster, and their fits differ 10x in cost), so the n > 2 jobs of a sharded round are dealt
    // out along the permutation k -> k * stride mod n: every shard gets the same mix. The stride is a prime that does not
    // divide n (n < 2^32 cannot be a multiple of all four).
    HPSDF_HD inline uint32_t dealStride(uint32_t n)
    {
        const uint32_t primes[4] = { 7919u, 7907u, 7901u, 7883u };
        for (int i = 0; i < 4; ++i)
            if (n % primes[i] != 0u) return primes[i];
        return 1u;
    }

    // What the host replay needs from a fit: the raw top-shell energy (Octree.cpp:1062-1069) and coeffs[0]
    // (the cell mean of the approximant up to NL[0][depth]^3, for the nearness weight).
    struct FitRecord
    {
        double rawErr;
        double c0;
    };

    // Per-degree projection tables in device memory: q[d][c*n + k] = w_k * P_c(xi_k) for the (4d+1)-point rule,
    // roots[d][k] = xi_k; bidx[idx] = a | b << 8 | c << 16 (BasisIndexValues, Utility.h:133-160).
    struct FitTablesDev
    {
        const double*   q[kMaxDegree + 1];
        const double*   roots[kMaxDegree + 1];
        const uint32_t* bidx;
    };

    // Device mesh (mesh.cpp builds it, mesh_eval.cuh traverses it)
    struct BvhNode            // 32 bytes
    {
        float    mn[3];
        uint32_t a;           // internal: left child index; leaf: first triangle slot
        float    mx[3];
        uint32_t b;           // internal: right child index; leaf: 0x80000000 | triangle count
    };

    struct DeviceMeshView
    {
        const BvhNode*  nodes;
        const void*     obb;          // 4 float4 per node: oriented box in the frame of the node's mean normal (mesh.cpp), see mesh_eval.cuh
        const void*     wide;         // 4-wide collapse of the same tree for meshSampleKernel: one 128-byte record per node = {4 child refs} + 4 x oriented box (frame code, centre, extents; mesh_build.cuh)
        const void*     triVerts;     // 3 float4 per triangle SLOT (BVH order): a, b, c; .w of a = original triangle index (bits)
        const float*    pseudo;       // 21 floats per ORIGINAL triangle: face normal, 3 edge normals (AB, BC, CA), 3 vertex normals (A, B, C)
        uint32_t        nTris, nNodes;
        float           inflate;      // absolute margin of the boxes against f32 rounding: 1e-5 of the mesh's size (mesh.cpp)
    };

    // Device SDF program (hpsdf_sdf_program with handles resolved to device pointers). Passed by value as a kernel parameter.
    struct DeviceTreeView;
    struct SdfInstrDev
    {
        uint32_t    op;
        uint32_t    pad;
        const void* handle;        // DeviceMeshView* / DeviceTreeView* in device memory, or nullptr
        double      p[8];
    };
    struct SdfProgramDev
    {
        uint32_t    n;
        uint32_t    pad;
        SdfInstrDev instr[HPSDF_PROGRAM_MAX_INSTR];
    };
#ifndef __CUDACC_RTC__
    // What launching a program's fits depends on: whether it samples a mesh or another octree (those fits sample F in a
    // kernel of its own, into scratch: fit_kernels.cuh) and its FLOPs per evaluation (6 for the root map + the operators).
    struct ProgramSummary
    {
        bool   samplesExt = false;
        double flopsPerEval = 6.0;
    };
    inline ProgramSummary summarizeProgram(const SdfProgramDev& prog)
    {
        ProgramSummary s;
        for (uint32_t i = 0; i < prog.n; ++i)
        {
            s.flopsPerEval += sdfOpFlops(prog.instr[i].op);
            s.samplesExt |= prog.instr[i].op == HPSDF_PRIM_MESH || prog.instr[i].op == HPSDF_PRIM_OCTREE;
        }
        return s;
    }
#endif

    // Leaf/internal node as the Query kernel reads it: 16 bytes, one LDG.128.
    struct QNode
    {
        uint32_t child;        // first child (8 consecutive), or 0xFFFFFFFF for a leaf
        uint32_t cstart;       // leaf: offset of its coefficients in the PADDED device store (even => 16-byte aligned)
        uint32_t degree;       // leaf degree; kInternalTag for internal nodes
        uint32_t depth;
    };

    struct DeviceTreeView
    {
        const QNode*    nodes;
        const double*   coeffs;      // padded store: every leaf starts at an even index
        const uint32_t* top;         // 4096 entries: node reached at depth <= 4 for each cell of the 16^3 grid (x + 16 y + 256 z)
        const uint32_t* bidx;        // BasisIndexValues of the tree's device (FitTablesDev::bidx)
        RootMap         map;
        uint32_t        nNodes;
    };
}
