/*
 * hpsdf.h — C ABI of the B200-native hp-adaptive SDF octree hot path.
 *
 * This is the drop-in boundary for ONE path of jw007123/hp-Adaptive-Signed-Distance-Field-Octree:
 * the octree build (fit / h-vs-p decision / refine / continuity solve) and batched Query, behind
 * the reference's public surface:
 *
 *     SDF::Config                               Include/HP/Config.h:12-43
 *     SDF::Octree::Create                       Include/HP/Octree.h:50,  Source/HP/Octree.cpp:312-352
 *     SDF::Octree::Query                        Include/HP/Octree.h:71,  Source/HP/Octree.cpp:662-702
 *     SDF::Octree::ToMemoryBlock                Include/HP/Octree.h:68,  Source/HP/Octree.cpp:424-456
 *     SDF::Octree::FromMemoryBlock              Include/HP/Octree.h:65,  Source/HP/Octree.cpp:403-421
 *     SDF::Octree::Clear / copy / GetRootAABB   Include/HP/Octree.h:44-47,62,81
 *     MemoryBlock                               Include/Utility/MemoryBlock.h:5-9
 *
 * Plain pointers and sizes only; no C++ or torch types. All entry points return hpsdf_status
 * (the reference only asserts); hpsdf_last_error() gives a thread-local message. There is NO CPU
 * fallback: every compute entry point fails with HPSDF_ERR_NO_DEVICE when no CUDA device is present.
 *
 * The C++ facade with the reference's names (SDF::Config, SDF::Octree, MemoryBlock) is
 * include/hpsdf.hpp of THIS repository; it forwards to these functions.
 */
#ifndef HPSDF_H
#define HPSDF_H

#ifndef HPSDF_NO_SYSTEM_HEADERS   /* defined by the library's run-time (NVRTC) compilation units only */
#include <stddef.h>
#include <stdint.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define HPSDF_API __attribute__((visibility("default")))
#else
#define HPSDF_API
#endif

/* ------------------------------------------------------------------------------------------ */
/* Status                                                                                       */
/* ------------------------------------------------------------------------------------------ */
typedef enum hpsdf_status
{
    HPSDF_OK              = 0,
    HPSDF_ERR_INVALID_ARG = 1,  /* null pointer, bad config (Config::IsValid asserts, Config.cpp:17-32) */
    HPSDF_ERR_NO_DEVICE   = 2,  /* no CUDA device / driver: there is no CPU path */
    HPSDF_ERR_CUDA        = 3,  /* a CUDA runtime call or kernel failed */
    HPSDF_ERR_BAD_BLOCK   = 4,  /* MemoryBlock does not parse (FromMemoryBlock asserts, Octree.cpp:405) */
    HPSDF_ERR_UNSUPPORTED = 5,  /* e.g. an SDF program this build cannot evaluate on device */
    HPSDF_ERR_COMM        = 6,  /* NCCL failure */
    HPSDF_ERR_OOM         = 7,
    HPSDF_ERR_MESH        = 8   /* mesh is not a closed manifold (Mesh::CreateHalfEdges fails, Mesh.cpp:121-128) */
} hpsdf_status;

HPSDF_API const char* hpsdf_status_string(hpsdf_status s);
HPSDF_API const char* hpsdf_last_error(void);
HPSDF_API const char* hpsdf_version(void);
/* Number of CUDA devices visible (0 when there is no driver); never fails. */
HPSDF_API int hpsdf_device_count(void);

/* ------------------------------------------------------------------------------------------ */
/* SDF::Config — byte image, LP64 (Include/HP/Config.h:12-43; offsets SURVEY.md App. B)         */
/* ------------------------------------------------------------------------------------------ */
enum
{
    HPSDF_NEARNESS_NONE        = 0,  /* Config::NearnessWeighting::None        */
    HPSDF_NEARNESS_POLYNOMIAL  = 1,  /* Config::NearnessWeighting::Polynomial  */
    HPSDF_NEARNESS_EXPONENTIAL = 2   /* Config::NearnessWeighting::Exponential */
};

typedef struct hpsdf_config
{
    uint8_t  nearness_type;           /* @0  nearnessWeighting.type      */
    uint8_t  _pad0[7];
    double   nearness_strength;       /* @8  nearnessWeighting.strength  */
    uint8_t  continuity_enforce;      /* @16 continuity.enforce          */
    uint8_t  _pad1[7];
    double   continuity_strength;     /* @24 continuity.strength         */
    uint8_t  enable_logging;          /* @32 enableLogging               */
    uint8_t  _pad2[7];
    double   target_error_threshold;  /* @40 targetErrorThreshold        */
    uint64_t thread_count;            /* @48 threadCount (u32 == unsigned long, Literals.h:9); ignored by the GPU build, kept in the blob */
    float    root_min[3];             /* @56 root.min()                  */
    float    root_max[3];             /* @68 root.max()                  */
} hpsdf_config;                       /* sizeof == 80 */

/* Config::Config() defaults (Config.cpp:5-14). */
HPSDF_API void hpsdf_config_default(hpsdf_config* cfg);
/* Config::IsValid() (Config.cpp:17-32) as a status instead of asserts. */
HPSDF_API hpsdf_status hpsdf_config_validate(const hpsdf_config* cfg);

/* ------------------------------------------------------------------------------------------ */
/* Build options that are compile-time constants or accidents of scheduling in the reference   */
/* (passed separately so sizeof(SDF::Config) stays 80).                                         */
/* ------------------------------------------------------------------------------------------ */
enum
{
    HPSDF_NEARNESS_EXACT_MEAN = 0,   /* mean of the approximant over the cell = c000 * 2^(3*depth/2): the deterministic
                                        limit of the reference's 100-sample std::rand() estimate (Octree.cpp:1209-1247) */
    HPSDF_NEARNESS_MC_COUNTER = 1,   /* the reference's estimator itself (mean of FApprox at 100 points of the cell) with the points
                                        from a counter-based generator instead of std::rand(): Philox4x32-10, key = nearness_seed,
                                        counter = (ix, iy, iz, depth | degree << 8 | sample << 16), u = (word >> 8) * 2^-24, point =
                                        min + (max - min) * u in f32 as AlignedBox::sample(). Reproducible for a given seed and
                                        independent of the schedule; for A/B runs against the literal reference. Device scheduler only. */
    HPSDF_TOTAL_REFERENCE     = 0,   /* totalCoeffError bookkeeping exactly as Octree.cpp:212,257,272,276 (sentinel 8^4*100) */
    HPSDF_TOTAL_EXACT_SUM     = 1,   /* sum of leaf errors recomputed without the sentinel bias (SURVEY.md F4) */
    HPSDF_CG_GUESS_COEFFS     = 0,
    HPSDF_CG_GUESS_REFERENCE  = 1
};

typedef struct hpsdf_comm hpsdf_comm;   /* one rank of a multi-GPU job, see hpsdf_comm_init */

typedef struct hpsdf_build_opts
{
    uint32_t struct_size;         /* = sizeof(hpsdf_build_opts) */
    uint32_t max_degree;          /* highest reachable basis degree; reference: BASIS_MAX_DEGREE-1 = 11 (Consts.h:7, Octree.cpp:600) */
    uint32_t max_depth;           /* reference: TREE_MAX_DEPTH = 10 (Consts.h:8) */
    uint32_t nearness_mode;       /* HPSDF_NEARNESS_EXACT_MEAN | HPSDF_NEARNESS_MC_COUNTER */
    uint32_t total_mode;          /* HPSDF_TOTAL_REFERENCE | HPSDF_TOTAL_EXACT_SUM */
    uint32_t cg_max_iterations;   /* 0 = 2n, Eigen's default */
    double   cg_tolerance;        /* relative residual; 0 = the reference's (double)1e-6f (Octree.cpp:1754) */
    int32_t  device;              /* CUDA device ordinal; -1 = current device */
    uint32_t speculate;           /* octaves (factors of 8 in error) below the guaranteed level whose jobs are pre-evaluated */
    uint32_t strict_order;        /* 1 = apply jobs in exactly the sequential greedy order (node numbering = the CPU checker's);
                                     0 = entries certain to be refined are applied as soon as their results are cached */
    hpsdf_comm* comm;             /* NULL = single GPU; else frontier jobs are sharded over the communicator's ranks */
    void*    stream;              /* cudaStream_t to run on; NULL = an internal non-blocking stream */
    uint32_t jit;                 /* closed-form programs: 0 = process default (hpsdf_set_jit / env HPSDF_JIT), 1 = compile the
                                     fit kernels for this program at run time (NVRTC, once per program and degree, ~0.3 s each,
                                     cached in memory), 2 = interpreted kernels. Mesh / octree programs are always interpreted. */
    uint32_t min_round_jobs;      /* a batched round evaluates at least this many refinement jobs when that many leaves are waiting
                                     (the next-largest errors beyond the guaranteed level); 0 = 512 for closed-form programs,
                                     128 for mesh / octree programs (device scheduler; the host replay uses 1 for those) */
    uint32_t scheduler;           /* 0 = the greedy loop (queue, h-vs-p decision, error bookkeeping, node allocation, job selection) runs
                                     on the device, one 112-byte header per round comes back; 1 = the loop is replayed on the host from
                                     16-byte fit records (round-1 implementation; also used when strict_order = 1) */
    uint32_t cg_guess;            /* initial guess of the continuity solve (M + lambda I) x = lambda c: 0 = the unconstrained coefficients c
                                     (the solution is c plus a small correction: 38 iterations instead of 71 on the README config, same
                                     stopping rule), 1 = the reference's own guess lambda c (solveWithGuess(oldCoeffs, oldCoeffs),
                                     Octree.cpp:1741, 1755) */
    uint64_t nearness_seed;       /* HPSDF_NEARNESS_MC_COUNTER: key of the sample-point generator */
} hpsdf_build_opts;

HPSDF_API void hpsdf_build_opts_default(hpsdf_build_opts* opts);
/* Process-wide default for hpsdf_build_opts.jit == 0 and for hpsdf_fit_batch / hpsdf_bench_frontier (off at start). */
HPSDF_API void hpsdf_set_jit(int on);

/* ------------------------------------------------------------------------------------------ */
/* Device SDF programs: what replaces the std::function<f64(Vector3d, u32)> argument of         */
/* Octree::Create (Octree.h:50) for SDFs that can live on the device.                           */
/* A program is a postfix (RPN) list: primitives push a distance, operators pop two, push one.  */
/* ------------------------------------------------------------------------------------------ */
typedef struct hpsdf_mesh   hpsdf_mesh;
typedef struct hpsdf_octree hpsdf_octree;

enum
{
    /* primitives; params in p[] (all f64 closed forms) */
    HPSDF_PRIM_SPHERE  = 1,   /* p[0..2] centre, p[3] radius:            |x-c| - r */
    HPSDF_PRIM_BOX     = 2,   /* p[0..2] centre, p[3..5] half extents                */
    HPSDF_PRIM_TORUS   = 3,   /* p[0..2] centre, p[3] R, p[4] r, p[5] axis (0,1,2)   */
    HPSDF_PRIM_CAPSULE = 4,   /* p[0..2] a, p[3..5] b, p[6] r                        */
    HPSDF_PRIM_PLANE   = 5,   /* p[0..2] unit normal, p[3] offset:       n.x - d     */
    HPSDF_PRIM_MESH    = 16,  /* handle = hpsdf_mesh*: float32 closest triangle + angle-weighted pseudonormal sign
                                 (Mesh::SignedDistanceAtPt, Source/Meshing/Mesh.cpp:54-63) */
    HPSDF_PRIM_OCTREE  = 17,  /* handle = hpsdf_octree*: Query of an existing tree (Octree.cpp:355-400 use this) */
    /* operators */
    HPSDF_OP_UNION     = 64,  /* min(a, b)      Octree::UnionSDF     Octree.cpp:368-371 */
    HPSDF_OP_INTERSECT = 65,  /* max(a, b)      Octree::IntersectSDF Octree.cpp:394-397 */
    HPSDF_OP_SUBTRACT  = 66,  /* max(a, -b)     a minus b                                */
    HPSDF_OP_NEGATE    = 67   /* -a                                                      */
};

#define HPSDF_PROGRAM_MAX_INSTR 16
#define HPSDF_PROGRAM_MAX_STACK 8

typedef struct hpsdf_sdf_instr
{
    uint32_t    op;
    uint32_t    _pad;
    const void* handle;     /* hpsdf_mesh* / hpsdf_octree* for MESH / OCTREE primitives, else NULL */
    double      p[8];
} hpsdf_sdf_instr;          /* sizeof == 80 */

typedef struct hpsdf_sdf_program
{
    uint32_t               n_instr;
    uint32_t               _pad;
    const hpsdf_sdf_instr* instr;
} hpsdf_sdf_program;

/* Evaluate a program at n points on the device (test hook for the evaluator; host pointers). */
HPSDF_API hpsdf_status hpsdf_sdf_eval(const hpsdf_sdf_program* prog, const double* xyz, size_t n, double* out, int device);

/* Device-resident triangle mesh + BVH; replaces Meshing::Mesh + Meshing::BVH as the SDF source
 * (Include/Meshing/Mesh.h:53-54, Include/Meshing/BVH.h:28).  vertices: n_vertices x 3 float32,
 * tri_indices: n_tris x 3 uint32 (CCW).  Fails with HPSDF_ERR_MESH if an edge has no twin. */
HPSDF_API hpsdf_status hpsdf_mesh_create(const float* vertices, size_t n_vertices,
                                         const uint32_t* tri_indices, size_t n_tris,
                                         int device, hpsdf_mesh** out);
/* Mesh::SignedDistanceAtPt batched, float32 throughout; host pointers. */
HPSDF_API hpsdf_status hpsdf_mesh_signed_distance(const hpsdf_mesh* mesh, const float* xyz, size_t n, float* out);
/* Mesh::CalculateMeshAABB (Mesh.cpp:66-84). */
HPSDF_API hpsdf_status hpsdf_mesh_aabb(const hpsdf_mesh* mesh, float mn[3], float mx[3]);
HPSDF_API void hpsdf_mesh_destroy(hpsdf_mesh* mesh);

/* ------------------------------------------------------------------------------------------ */
/* SDF::Octree                                                                                  */
/* ------------------------------------------------------------------------------------------ */

/* Octree::Create (Octree.cpp:312-352). Blocks the calling thread; drives the GPU on opts->stream. */
HPSDF_API hpsdf_status hpsdf_create(const hpsdf_config* cfg, const hpsdf_build_opts* opts,
                                    const hpsdf_sdf_program* prog, hpsdf_octree** out);

/* Octree::Query (Octree.cpp:662-702) for n points, xyz = n x 3 f64 (AoS), out = n f64, HOST pointers.
 * Points outside the root give DBL_MAX (Octree.cpp:668-671). Thread-safe on a finished tree. */
HPSDF_API hpsdf_status hpsdf_query(const hpsdf_octree* tree, const double* xyz, size_t n, double* out);
/* Same with DEVICE pointers, asynchronous on `stream` (cudaStream_t; NULL = legacy default stream). The tree's device must be the
 * current device. d_xyz needs 8-byte alignment only (a 16-byte aligned array takes the vectorised load path). */
HPSDF_API hpsdf_status hpsdf_query_device(const hpsdf_octree* tree, const double* d_xyz, size_t n, double* d_out, void* stream);
/* Octree::QueryWithGradient (Octree.cpp:749-789, 904-985): value + unit central-difference gradient. */
HPSDF_API hpsdf_status hpsdf_query_with_gradient(const hpsdf_octree* tree, const double* xyz, size_t n, double* out, double* unit_grad);

/* Value and exact derivatives of the field hpsdf_query evaluates (DESIGN.md §13; no counterpart in the reference). For each
 * point, Query's leaf and local coordinate u (same root map, f32 containment test and descent) give F(x) = P_leaf(u(x)),
 * u_a = (p_a - c_a) 2^(depth+1), p_a = (x_a - centre_a) invSizes_a with Query's f32-rounded invSizes; s_a = 2^(depth+1) invSizes_a.
 *   value[i]        = hpsdf_query's value, bit for bit (DBL_MAX outside the root);
 *   grad[3i + a]    = dP/du_a s_a: the gradient in user space, NOT normalised;
 *   hess[6i + k]    = d2P/du_a du_b s_a s_b in the order xx, xy, xz, yy, yz, zz; hess may be NULL (not computed).
 * Outside the root grad and hess are 0. F is not continuous across leaf faces: at a point on a face the derivatives are
 * those of the leaf Query picks (one-sided). xyz = n x 3 f64 (AoS), HOST pointers; blocks the calling thread.
 * HPSDF_ERR_NO_DEVICE without a GPU; HPSDF_ERR_INVALID_ARG for a null tree, or a null xyz, value or grad when n > 0. */
HPSDF_API hpsdf_status hpsdf_query_derivatives(const hpsdf_octree* tree, const double* xyz, size_t n, double* value, double* grad,
                                               double* hess);
/* Same with DEVICE pointers, asynchronous on `stream`; the current device must be the tree's (HPSDF_ERR_INVALID_ARG otherwise).
 * d_xyz needs 8-byte alignment only. */
HPSDF_API hpsdf_status hpsdf_query_derivatives_device(const hpsdf_octree* tree, const double* d_xyz, size_t n, double* d_value,
                                                      double* d_grad, double* d_hess, void* stream);

/* Octree::QueryRay (Octree.cpp:705-746, Ray.cpp:5-65) for n rays: origins / directions n x 3 f64, hit n bytes (1 = the march
 * reached a field value below 1e-4 within 200 steps and t_max), t n f64 (the reference stores the last field value there).
 * Statement-by-statement mirror of the reference, see query_kernels.cuh for what that implies outside the default root box. */
HPSDF_API hpsdf_status hpsdf_query_ray(const hpsdf_octree* tree, const double* origins, const double* directions, size_t n, double t_max,
                                       unsigned char* hit, double* t);

/* First crossing of the level set F = iso along n rays x(t) = o + t*d, t in [t_min, t_max] (user space, d need not be
 * unit; t is in units of d). F is the tree's own piecewise polynomial field: Query's leaves and coefficients, DBL_MAX
 * outside the root box. t_hit[i] = the smallest t at which F <= iso, or +INFINITY for a miss. normals (may be NULL):
 * the unit gradient of the hit leaf's polynomial at t_hit in user space, pointing to increasing F; (0,0,0) on a miss
 * or a vanishing gradient. Each leaf's polynomial along the ray is solved exactly (DESIGN.md §12): no step size, no
 * Lipschitz assumption, thin parts and jumps across leaf faces are found; any root box works. This, not
 * hpsdf_query_ray (the reference's mirror), is the ray query to use.
 * HPSDF_ERR_INVALID_ARG: null pointers when n > 0 (normals may be NULL), non-finite t_min or iso, t_max < t_min or NaN
 * (t_max = +inf is allowed). A zero or non-finite direction or a non-finite origin is a miss. Blocks the calling thread. */
HPSDF_API hpsdf_status hpsdf_raycast(const hpsdf_octree* tree, const double* origins, const double* directions, size_t n,
                                     double t_min, double t_max, double iso, double* t_hit, double* normals);
/* Same with DEVICE pointers, asynchronous on `stream`; the current device must be the tree's (as hpsdf_query_device). */
HPSDF_API hpsdf_status hpsdf_raycast_device(const hpsdf_octree* tree, const double* d_origins, const double* d_directions,
                                            size_t n, double t_min, double t_max, double iso, double* d_t_hit,
                                            double* d_normals, void* stream);

/* The level set F = iso of the tree as a triangle mesh: marching tetrahedra over a uniform grid of
 * resolution[0] x resolution[1] x resolution[2] cells spanning [box_min, box_max] (both NULL = the root box).
 * Grid values are Query values (DBL_MAX outside the root). Vertices: n_vertices x 3 float32, triangles:
 * n_triangles x 3 uint32, counter-clockwise seen from the side where F >= iso. Both arrays are malloc()ed;
 * the CALLER free()s them (as hpsdf_to_memory_block). An empty result gives 0, 0 and NULL pointers.
 * Blocks the calling thread; runs on the tree's device.
 *
 * Grid point (i,j,k) is box_min + idx * h per axis, h = (box_max - box_min) / resolution, each operation rounded in f64;
 * a corner is inside when its value is below iso. Every cell is cut into the six Kuhn tetrahedra along its 0-7 diagonal.
 * Vertices are ordered by the grid point that owns their edge (its lower end), then by edge direction; triangles by cell,
 * tetrahedron and position (DESIGN.md §11 has the full contract). When no grid point on the box's boundary faces is
 * inside, the mesh is a closed, oriented 2-manifold with every vertex used (hpsdf_mesh_create accepts it); a surface that
 * crosses the box leaves the mesh open there. A grid value exactly equal to iso puts vertices on that grid point, so
 * zero-area triangles can appear. Resolutions are 1..1024; HPSDF_ERR_UNSUPPORTED when either count exceeds 2^32 - 1. */
HPSDF_API hpsdf_status hpsdf_extract_isosurface(const hpsdf_octree* tree, const uint32_t resolution[3],
                                                const double box_min[3], const double box_max[3], double iso,
                                                size_t* n_vertices, float** vertices,
                                                size_t* n_triangles, uint32_t** tri_indices);

/* Octree::ToMemoryBlock (Octree.cpp:424-456): *ptr is malloc()ed, the CALLER free()s it. LP64 layout. */
HPSDF_API hpsdf_status hpsdf_to_memory_block(const hpsdf_octree* tree, size_t* size, void** ptr);
/* Octree::FromMemoryBlock (Octree.cpp:403-421): copies; the caller keeps ownership of the block. */
HPSDF_API hpsdf_status hpsdf_from_memory_block(const void* ptr, size_t size, int device, hpsdf_octree** out);
/* Octree copy constructor (Octree.cpp:24-45). */
HPSDF_API hpsdf_status hpsdf_clone(const hpsdf_octree* tree, hpsdf_octree** out);
/* Octree::GetRootAABB (Octree.cpp:106-109). */
HPSDF_API hpsdf_status hpsdf_get_root_aabb(const hpsdf_octree* tree, float mn[3], float mx[3]);
/* The Config the tree was created with (what the reference keeps in Octree::config, Octree.h:91, and writes at the end of a
 * MemoryBlock) and the CUDA device its storage lives on. */
HPSDF_API hpsdf_status hpsdf_get_config(const hpsdf_octree* tree, hpsdf_config* cfg);
HPSDF_API hpsdf_status hpsdf_get_device(const hpsdf_octree* tree, int* device);
/* Octree::~Octree / Clear (Octree.cpp:15-21, 459-471). */
HPSDF_API void hpsdf_destroy(hpsdf_octree* tree);

/* Counters of the last Create on this tree (the reference only printf()s, Octree.cpp:292-296). */
typedef struct hpsdf_build_stats
{
    uint64_t n_nodes, n_leaves, n_coeffs;
    uint64_t rounds;              /* batched evaluation rounds */
    uint64_t jobs_evaluated;      /* refinement jobs computed on the device (incl. speculative ones never applied) */
    uint64_t jobs_applied_p, jobs_applied_h;
    uint64_t fits_evaluated;      /* FitPolynomial-equivalents computed (coarse fit, child fit or p-fit) */
    uint64_t sdf_evals;           /* SDF samples evaluated */
    uint64_t kernel_launches;     /* kernels of this library launched by the build */
    double   algorithmic_flops;   /* sum-factorised FLOPs of those fits incl. sdf_evals * sdf_flops_per_eval (SURVEY.md §8d formula) */
    double   sdf_flops_per_eval;  /* c_F of the SDF program: closed-form FLOPs per sample, sqrt and divide counted as one */
    double   total_error;         /* totalCoeffError at termination (reference bookkeeping or exact, per total_mode) */
    double   exact_total_error;   /* plain sum of leaf errors at termination */
    double   cut_margin;          /* (threshold - total)/threshold at termination: small = near-threshold stop */
    double   fit_kernel_ms;       /* device time in fit kernels (CUDA events on the build stream) */
    double   continuity_ms;       /* wall time of the continuity post-process: face enumeration + assembly + CG */
    double   continuity_enum_ms, continuity_assembly_ms, continuity_cg_ms;   /* its parts: host face walk; emit + sort + CSR; CG */
    double   host_replay_ms;      /* host time in the greedy replay */
    double   host_select_ms;      /* host time choosing which leaves to evaluate each round */
    double   host_tasks_ms;       /* host time building fit task lists */
    double   device_wait_ms;      /* host time blocked on the build stream (kernels + copies) */
    double   pack_ms, finalize_ms;/* ReallocCoeffs gather; Query structures */
    double   total_ms;            /* wall time of hpsdf_create */
    uint64_t cg_iterations;
    double   cg_relative_residual;
    uint64_t near_tie_decisions;  /* h-vs-p decisions with |pImp-hImp| <= 1e-9*max(|pImp|,|hImp|) (see hpsdf_get_decision_log) */
} hpsdf_build_stats;

HPSDF_API hpsdf_status hpsdf_get_build_stats(const hpsdf_octree* tree, hpsdf_build_stats* stats);

/* Near-threshold refinement decisions of the last Create, with their margins (north_star: "any
 * near-threshold refinement divergence logged with its error margin"). */
typedef struct hpsdf_decision_log_entry
{
    uint64_t node_idx;
    uint32_t depth, degree;
    float    centre[3];           /* cell centre in the internal unit cube */
    uint32_t chose_p;             /* 1 = p-refinement, 0 = h-refinement */
    uint32_t kind;                /* 0 = h/p near-tie, 1 = last job applied before the termination cut,
                                     2 / 3 = member of the group of equal-error leaves the cut falls into: refined / left unrefined */
    double   p_improvement, h_improvement;
    double   relative_margin;
} hpsdf_decision_log_entry;

HPSDF_API size_t hpsdf_get_decision_log(const hpsdf_octree* tree, hpsdf_decision_log_entry* out, size_t capacity);

/* Every refinement applied by the last Create, in order (what enableLogging printf()s one line for, Octree.cpp:292-296):
 * lets a caller diff two builds job by job. */
typedef struct hpsdf_apply_log_entry
{
    uint64_t node_idx;
    uint32_t kind;                /* 0 = P (degree + 1), 1 = H (split into 8) */
    uint32_t degree;              /* degree before the job */
    double   initial_err, new_err;/* new_err: P: the new error; H: the largest child error */
    double   p_improvement, h_improvement;
    double   total_after;         /* totalCoeffError after applying it */
} hpsdf_apply_log_entry;

HPSDF_API size_t hpsdf_get_apply_log(const hpsdf_octree* tree, hpsdf_apply_log_entry* out, size_t capacity);

/* ------------------------------------------------------------------------------------------ */
/* Kernel-level entry points (benchmarks / parity of single stages)                             */
/* ------------------------------------------------------------------------------------------ */

/* FitPolynomial (Octree.cpp:1007-1093) for a batch of independent cells, from scratch at `degree`:
 * cells = n x 4 float32 {centre x,y,z, half size} in the internal unit cube; depth[i] = tree depth of cell i
 * (selects NormalisedLengths[.][depth], Utility.h:63-78).  coeffs_out = n x N_degree f64 in BasisIndexValues
 * order (Utility.h:133-160), raw_err_out = n f64 (top-shell energy, no nearness weight). Host pointers.
 * elapsed_ms (optional) = device time of the fit kernel alone. */
HPSDF_API hpsdf_status hpsdf_fit_batch(const hpsdf_config* cfg, const hpsdf_sdf_program* prog,
                                       const float* cells, const uint8_t* depth, size_t n, uint32_t degree,
                                       double* coeffs_out, double* raw_err_out, int device, float* elapsed_ms);

/* A synthetic frontier of refinement jobs (SURVEY.md §8d): every cell of a uniform grid at `grid_depth`
 * evaluated as a job at degree p (8 child fits @p + 1 p-fit @p+1), `repeats` timed launches after one
 * warm-up.  Returns the average device milliseconds per launch, the jobs and fits per launch and the
 * algorithmic FLOPs per launch. */
typedef struct hpsdf_frontier_bench
{
    double   ms_per_launch;
    uint64_t jobs, fits, sdf_evals;
    double   algorithmic_flops;     /* contraction FLOPs + sdf_evals * sdf_flops_per_eval */
    double   sdf_flops_per_eval;
    double   checksum;              /* sum of all error outputs, so the work cannot be elided */
} hpsdf_frontier_bench;

HPSDF_API hpsdf_status hpsdf_bench_frontier(const hpsdf_config* cfg, const hpsdf_sdf_program* prog,
                                            uint32_t grid_depth, uint32_t degree, uint32_t repeats,
                                            int device, void* stream, hpsdf_frontier_bench* out);

/* Generates the straight-line CUDA of `prog` (closed-form primitives only) and compiles the degree-`degree` fit kernel for
 * sm_100a with NVRTC, without touching a device: the build check of the run-time specialiser (hpsdf_build_opts.jit).
 * source_out (may be NULL) receives the generated translation unit, cubin_bytes (may be NULL) the size of the cubin. */
HPSDF_API hpsdf_status hpsdf_jit_compile_check(const hpsdf_sdf_program* prog, uint32_t degree, char* source_out, size_t source_cap,
                                               size_t* cubin_bytes);

/* The synthetic Query workload of BASELINE config 5 (SURVEY.md 8d): n points uniform in [lo, hi) written to d_xyz (n x 3 f64,
 * DEVICE pointer, current device, asynchronous on `stream`), point i = Philox4x32-10(key = seed, counter = first_index + i),
 * 53-bit mantissas. A point depends only on (seed, global index): any sharding or chunking evaluates the same set. */
HPSDF_API hpsdf_status hpsdf_uniform_points_device(uint64_t seed, uint64_t first_index, size_t n, const double lo[3], const double hi[3],
                                                   double* d_xyz, void* stream);

/* FP64 FMA peak of the device measured with a register-resident DFMA chain (TFLOP/s); the roofline
 * denominator for fitting, which MEASURED_PEAKS.json does not hold. */
HPSDF_API hpsdf_status hpsdf_measure_fp64_peak(int device, void* stream, double* tflops);

/* ------------------------------------------------------------------------------------------ */
/* Multi-GPU: one process per GPU; the frontier is sharded over ranks and the per-round job     */
/* records are all-gathered with NCCL so every rank replays the same greedy order.              */
/* ------------------------------------------------------------------------------------------ */
#define HPSDF_COMM_ID_BYTES 128
/* rank 0 calls this and ships the 128 bytes to the other ranks by any means (e.g. torch.distributed). */
HPSDF_API hpsdf_status hpsdf_comm_get_unique_id(void* id_out);
HPSDF_API hpsdf_status hpsdf_comm_init(const void* id, int rank, int world_size, int device, hpsdf_comm** out);
HPSDF_API void hpsdf_comm_destroy(hpsdf_comm* comm);
/* Contiguous shard [begin, end) of n items owned by `rank` (pure host function). */
HPSDF_API void hpsdf_shard_range(size_t n, int rank, int world_size, size_t* begin, size_t* end);

#ifdef __cplusplus
}
#endif
#endif /* HPSDF_H */
