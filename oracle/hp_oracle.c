/*
 * oracle/hp_oracle.c — plain-C CPU restatement of the reference's hp-adaptive SDF octree hot path.
 *
 * TEST INFRASTRUCTURE ONLY. Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may load the
 * library built from this file (oracle/_build/libhporacle.so). The product path never links or calls it.
 *
 * What it restates (file:line are relative to /root/reference):
 *   tables                       Include/HP/Utility.h:14-196, Include/HP/Legendre.h (regenerated, see tools/gen_gl_tables.py)
 *   CreateRoot/Subdivide/Corner  Source/HP/Octree.cpp:792-801, 1096-1128
 *   UniformlyRefine              Source/HP/Octree.cpp:112-191
 *   FitPolynomial / LpX          Source/HP/Octree.cpp:988-1093
 *   job (h/p estimate, decision) Source/HP/Octree.cpp:558-659, 804-856
 *   greedy scheduler             Source/HP/Octree.cpp:194-309 — as the DETERMINISTIC schedule: strict greedy, window 1,
 *                                termination checked after every applied job; nearness weight from the exact cell mean
 *                                instead of 100 std::rand() samples (Octree.cpp:1209-1247); SURVEY.md F3-F5.
 *   ReallocCoeffs                Source/HP/Octree.cpp:474-555
 *   Query / FApprox              Source/HP/Octree.cpp:662-702, 859-901
 *   QueryWithGradient            Source/HP/Octree.cpp:749-789, 904-985
 *   continuity                   Source/HP/Octree.cpp:1250-1762 (face enumeration, analytic + numeric blocks, (M+lambda I)x = lambda c)
 *   To/FromMemoryBlock           Source/HP/Octree.cpp:403-456 (LP64 layout, SURVEY.md App. B)
 *
 * Pinning: built with -ffp-contract=off and the reference's operation order, the fit, the job arithmetic and the heap
 * are BIT-IDENTICAL to oracle/_ref/libhpref.so's deterministic driver (reference sources + ref_driver.cpp); tests/
 * test_oracle_vs_ref.py asserts equality of apply logs, coefficients and query values, and tests/golden/ holds
 * vectors generated from the reference itself. The CG iterate is NOT pinned (Eigen's IncompleteCholesky is unpinned
 * third-party code absent here): parity is on the converged solution.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <stdio.h>
#include <float.h>
#include <time.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#include "../include/hpsdf.h"
#include "sdf_cpu.h"
#include "hp_oracle_tables.h"
#include "hp_oracle_mesh.h"

#define MAXDEG 12           /* BASIS_MAX_DEGREE, Consts.h:7 */
#define MAXDEPTH 10         /* TREE_MAX_DEPTH,  Consts.h:8 */
#define INTERNAL_TAG 13     /* BASIS_MAX_DEGREE + 1, Node.cpp:12 */
#define NO_CHILD UINT64_MAX /* childIdx = -1, Node.cpp:8 */
#define INITIAL_NODE_ERR 100.0

/* ---- tables (Utility.h) --------------------------------------------------------------------------------- */
/* LegendreCoeffientCount (Utility.h:87-106): (u32)((1.0/6.0)*(i+1)*(i+2)*(i+3)) — the f64 product truncates to 83 (not 84)
 * for i = 6; the quirk is part of the MemoryBlock contract (a degree-6 leaf stores 83 coefficients). */
static uint32_t COUNT[MAXDEG + 1];
static double   NL[MAXDEG + 1][MAXDEPTH + 1];   /* NormalisedLengths, Utility.h:63-78 */
static double   REC[MAXDEG + 1][2];             /* LegendreCoefficent, Utility.h:112-127 */
static uint32_t BIDX[455][3];                   /* BasisIndexValues, Utility.h:133-160 */
static uint32_t FACE[3][4][2];                  /* SharedFaceLookup, Utility.h:166-196 */
/* GL rules in the reference's node order: ascending |x|, negative root first (Legendre.h) */
static double   ROOTS[2080], WEIGHTS[2080];
static int      g_init = 0;

static double sqrt_newton(double x) { double g = x; for (int i = 0; i < 100; ++i) g = 0.5 * (g + x / g); return g; }   /* Utility.h:25-35 */

void hporacle_init(void)
{
    if (g_init) return;
    const double f = 1.0 / 6.0;
    for (uint32_t i = 0; i <= MAXDEG; ++i)
    {
        COUNT[i] = (uint32_t)(f * (i + 1) * (i + 2) * (i + 3));
        for (uint32_t j = 0; j <= MAXDEPTH; ++j)
        {
            double pw = 1.0;
            for (uint32_t k = 0; k < j; ++k) pw = 2.0 * pw;
            NL[i][j] = sqrt_newton((2.0 * i + 1.0) * pw);
        }
        REC[i][0] = i ? (2.0 * i - 1.0) / i : 0.0;
        REC[i][1] = i ? (i - 1.0) / i : 0.0;
    }
    uint32_t n = 0;
    for (uint32_t p = 0; p <= MAXDEG; ++p)
        for (uint32_t i = 0; i <= p; ++i)
            for (uint32_t j = 0; j <= p - i; ++j) { BIDX[n][0] = i; BIDX[n][1] = j; BIDX[n][2] = p - i - j; n++; }
    for (uint32_t d = 0; d < 3; ++d)
    {
        uint32_t k = 0;
        for (uint32_t c = 0; c < 8; ++c) if (!(c & (1u << d))) { FACE[d][k][0] = c; FACE[d][k][1] = c | (1u << d); k++; }
    }
    /* Re-order each ascending rule to the reference table's order (it only affects summation order, i.e. the last
     * ulp): zero first, then +-pairs by ascending |x|, negative root first. Two rules of the reference's table list
     * their pairs in another order (n = 6: 2nd,1st,3rd; n = 9: 3rd,4th,1st,2nd) — observed through hpref_tables(),
     * reproduced here so the degree-2 coarse fits (9-point rule) are bit-identical. */
    static const uint32_t pairOrder6[3] = { 1, 0, 2 }, pairOrder9[4] = { 2, 3, 0, 1 };
    for (uint32_t r = 1; r <= 64; ++r)
    {
        const uint32_t o = r * (r - 1) / 2;
        uint32_t w = 0;
        if (r & 1) { ROOTS[o] = hporacle_gl_roots[o + r / 2]; WEIGHTS[o] = hporacle_gl_weights[o + r / 2]; w = 1; }
        for (uint32_t kk = 0; kk < r / 2; ++kk)
        {
            const uint32_t k = r == 6 ? pairOrder6[kk] : r == 9 ? pairOrder9[kk] : kk;
            const uint32_t lo = o + r / 2 - 1 - k, hi = o + (r + 1) / 2 + k;
            ROOTS[o + w] = hporacle_gl_roots[lo]; WEIGHTS[o + w] = hporacle_gl_weights[lo]; w++;
            ROOTS[o + w] = hporacle_gl_roots[hi]; WEIGHTS[o + w] = hporacle_gl_weights[hi]; w++;
        }
    }
    g_init = 1;
}

void hporacle_tables(double* nl, uint32_t* counts, uint32_t* bidx, double* rec, double* roots, double* weights, uint32_t* face)
{
    hporacle_init();
    memcpy(nl, NL, sizeof(NL)); memcpy(counts, COUNT, sizeof(COUNT)); memcpy(bidx, BIDX, sizeof(BIDX));
    memcpy(rec, REC, sizeof(REC)); memcpy(roots, ROOTS, sizeof(ROOTS)); memcpy(weights, WEIGHTS, sizeof(WEIGHTS));
    memcpy(face, FACE, sizeof(FACE));
}

/* LpX, Octree.cpp:988-1004 */
static double LpX(uint32_t p, double x)
{
    double m2 = 0.0, m1 = 1.0, l = 1.0;
    for (uint32_t i = 1; i <= p; ++i) { l = REC[i][0] * x * m1 - REC[i][1] * m2; m2 = m1; m1 = l; }
    return l;
}

/* ---- tree ------------------------------------------------------------------------------------------------ */
typedef struct { float mn[3], mx[3]; } Box;

typedef struct
{
    uint64_t child;       /* NO_CHILD for a leaf */
    Box      aabb;
    double*  coeffs;      /* build-time ownership; NULL after packing */
    uint64_t cstart;      /* offset into the packed store after ReallocCoeffs */
    uint8_t  degree;      /* INTERNAL_TAG for internal nodes */
    uint8_t  depth;
} Node;

typedef struct { uint64_t idx; double err; } HeapItem;

typedef struct
{
    uint64_t node; uint32_t kind, degree; double initialErr, newErr, pImp, hImp, totalAfter;
} ApplyRecord;

typedef struct
{
    hpsdf_config     cfg;
    hpsdf_sdf_instr* prog; uint32_t nprog;
    hporacle_ext_eval ext;
    double rootCentre[3], rootSizes[3], rootInvSizes[3];
    Node*  nodes; size_t nNodes, capNodes;
    double* store; size_t nCoeffs;
    HeapItem* heap; size_t nHeap, capHeap;
    ApplyRecord* log; size_t nLog, capLog;
    double seconds, continuitySeconds, finalTotal, cgError;
    uint64_t fits, jobs, appliedP, appliedH, cgIterations;
} Tree;

static void box_center(const Box* b, float c[3]) { for (int i = 0; i < 3; ++i) c[i] = (b->mn[i] + b->mx[i]) / 2.0f; }   /* AlignedBox::center */

static void set_root_mapping(Tree* t)
{
    /* Octree.cpp:322-324 / 419-420: centre and sizes in f32, inverse sizes computed IN f32, all widened */
    for (int i = 0; i < 3; ++i)
    {
        const float c = (t->cfg.root_min[i] + t->cfg.root_max[i]) / 2.0f;
        const float s = t->cfg.root_max[i] - t->cfg.root_min[i];
        t->rootCentre[i] = (double)c; t->rootSizes[i] = (double)s; t->rootInvSizes[i] = (double)(1.0f / s);
    }
}

/* F of Octree.cpp:325-328: the user SDF composed with the unit-cube -> root map */
static double eval_F(const Tree* t, const double u[3])
{
    const double x[3] = { u[0] * t->rootSizes[0] + t->rootCentre[0], u[1] * t->rootSizes[1] + t->rootCentre[1], u[2] * t->rootSizes[2] + t->rootCentre[2] };
    return hporacle_sdf_eval(t->prog, t->nprog, x, t->ext);
}

static uint64_t push_node(Tree* t)
{
    if (t->nNodes == t->capNodes) { t->capNodes = t->capNodes ? 2 * t->capNodes : 8192; t->nodes = (Node*)realloc(t->nodes, t->capNodes * sizeof(Node)); }
    Node* n = &t->nodes[t->nNodes];
    memset(n, 0, sizeof(*n));
    n->child = NO_CHILD; n->degree = INTERNAL_TAG; n->depth = MAXDEPTH + 1;          /* Node.cpp:6-15 */
    for (int i = 0; i < 3; ++i) { n->aabb.mn[i] = FLT_MAX; n->aabb.mx[i] = -FLT_MAX; }
    return t->nNodes++;
}

/* CornerAABB, Octree.cpp:1096-1112 */
static Box corner_aabb(const Box* b, uint32_t i)
{
    Box c = *b;
    for (int d = 0; d < 3; ++d)
    {
        const float mid = (b->mx[d] + b->mn[d]) * 0.5f;
        if (i & (1u << d)) c.mn[d] = mid; else c.mx[d] = mid;
    }
    return c;
}

/* Subdivide, Octree.cpp:1115-1128 */
static void subdivide(Tree* t, uint64_t idx)
{
    t->nodes[idx].child = t->nNodes;
    for (uint32_t i = 0; i < 8; ++i)
    {
        const uint64_t c = push_node(t);
        t->nodes[c].aabb  = corner_aabb(&t->nodes[idx].aabb, i);
        t->nodes[c].depth = t->nodes[idx].depth + 1;
    }
}

/* std::priority_queue<pair<u32,f64>, vector, PriorityQueuePredicate> (Octree.h:95-102): a max-heap on err with the
 * libstdc++ heap algorithms (push_heap = sift up; pop_heap = move the hole down to a leaf along the larger child, then
 * sift the displaced last element up), so equal keys pop in the same order as the reference's nodeQueue. */
static int heap_less(const HeapItem* a, const HeapItem* b) { return a->err < b->err; }

static void heap_sift_up(HeapItem* h, size_t hole, size_t top, HeapItem v)
{
    while (hole > top)
    {
        const size_t parent = (hole - 1) / 2;
        if (!heap_less(&h[parent], &v)) break;
        h[hole] = h[parent]; hole = parent;
    }
    h[hole] = v;
}

static void heap_push(Tree* t, uint64_t idx, double err)
{
    if (t->nHeap == t->capHeap) { t->capHeap = t->capHeap ? 2 * t->capHeap : 8192; t->heap = (HeapItem*)realloc(t->heap, t->capHeap * sizeof(HeapItem)); }
    const HeapItem v = { idx, err };
    heap_sift_up(t->heap, t->nHeap, 0, v);
    t->nHeap++;
}

static HeapItem heap_pop(Tree* t)
{
    HeapItem* h = t->heap;
    const HeapItem top = h[0];
    const size_t len = --t->nHeap;       /* elements that stay */
    if (len == 0) return top;
    const HeapItem v = h[len];
    size_t hole = 0, second = 0;
    while (second < (len - 1) / 2)
    {
        second = 2 * (second + 1);
        if (heap_less(&h[second], &h[second - 1])) second--;
        h[hole] = h[second]; hole = second;
    }
    if ((len & 1) == 0 && second == (len - 2) / 2)
    {
        second = 2 * (second + 1);
        h[hole] = h[second - 1]; hole = second - 1;
    }
    heap_sift_up(h, hole, 0, v);
    return top;
}

/* CreateRoot + UniformlyRefine, Octree.cpp:792-801, 112-191: pre-order DFS, Subdivide on first visit, children 0..7;
 * depth-4 cells get degree 0 and enter the queue with err = 100 in visiting order. */
static void refine_uniform(Tree* t, uint64_t idx, uint32_t depth)
{
    if (depth < 4)
    {
        subdivide(t, idx);
        const uint64_t c = t->nodes[idx].child;
        for (uint32_t i = 0; i < 8; ++i) refine_uniform(t, c + i, depth + 1);
    }
    else
    {
        t->nodes[idx].coeffs = (double*)malloc(sizeof(double) * COUNT[2]);
        t->nodes[idx].degree = 0;
        heap_push(t, idx, INITIAL_NODE_ERR);
    }
}

static void create_root_and_coarse_grid(Tree* t)
{
    const uint64_t r = push_node(t);
    t->nodes[r].depth = 0;
    for (int i = 0; i < 3; ++i) { t->nodes[r].aabb.mn[i] = -0.5f; t->nodes[r].aabb.mx[i] = 0.5f; }
    subdivide(t, 0);
    for (uint32_t i = 0; i < 8; ++i) refine_uniform(t, 1 + i, 1);
}

/* FitPolynomial, Octree.cpp:1007-1093, nearness None (raw top-shell energy). Same loop nest, sample order and operation
 * order as the reference; only LpX(a, root) is hoisted into a table (identical values). */
static double fit_polynomial(const Tree* t, double* coeffs, uint32_t degreeIn, const Box* aabb, uint32_t degree, uint32_t depth)
{
    const uint32_t start = degreeIn > 0 ? COUNT[degreeIn] : 0, end = COUNT[degree];
    const uint32_t n = 4 * degree + 1, gq = (4 * degree) * (4 * degree + 1) / 2;      /* SumToN[4*degree], Octree.cpp:1016 */
    double scale[3], centre[3];
    float cf[3];
    box_center(aabb, cf);
    for (int i = 0; i < 3; ++i) { scale[i] = (double)(aabb->mx[i] - aabb->mn[i]) * 0.5; centre[i] = (double)cf[i]; }
    const double scalesMult = scale[0] * (scale[1] * scale[2]);
    double (*L)[MAXDEG + 1] = (double (*)[MAXDEG + 1])malloc(sizeof(double) * n * (MAXDEG + 1));
    for (uint32_t i = 0; i < n; ++i) for (uint32_t a = 0; a <= degree; ++a) L[i][a] = LpX(a, ROOTS[gq + i]);

    memset(coeffs + start, 0, (end - start) * sizeof(double));
    for (uint32_t i = 0; i < n; ++i)
        for (uint32_t j = 0; j < n; ++j)
            for (uint32_t k = 0; k < n; ++k)
            {
                const double u[3] = { ROOTS[gq + i] * scale[0] + centre[0], ROOTS[gq + j] * scale[1] + centre[1], ROOTS[gq + k] * scale[2] + centre[2] };
                const double wprod = WEIGHTS[gq + i] * (WEIGHTS[gq + j] * WEIGHTS[gq + k]);
                const double fs = scalesMult * wprod * eval_F(t, u);
                for (uint32_t c = start; c < end; ++c)
                {
                    double lp = 1.0;
                    lp *= L[i][BIDX[c][0]]; lp *= NL[BIDX[c][0]][depth];
                    lp *= L[j][BIDX[c][1]]; lp *= NL[BIDX[c][1]][depth];
                    lp *= L[k][BIDX[c][2]]; lp *= NL[BIDX[c][2]][depth];
                    coeffs[c] += lp * fs;
                }
            }
    free(L);
    double err = 0.0;
    for (uint32_t i = 0; i < end; ++i)
        if (BIDX[i][0] + BIDX[i][1] + BIDX[i][2] == degree) err += coeffs[i] * coeffs[i];
    return err;
}

/* ---- nearness weight (CalculatePolyWeighting / CalculateExpWeighting, Octree.cpp:1209-1247) ----------------------------
 * The reference averages FApprox over 100 points from aabb_.sample(), i.e. std::rand(): not reproducible. Two
 * deterministic statements of it:
 *   exact mean (default): the cell mean of the approximant is coeffs[0] * NL[0][depth]^3 (orthonormal basis) — the limit
 *                         of the estimate for many samples;
 *   mc_counter(seed):     the reference's estimator itself, 100 samples, with the sample points drawn from a counter-based
 *                         generator instead of std::rand(): Philox4x32-10, key = seed, counter = (ix, iy, iz,
 *                         depth | degree << 8 | sample << 16) with (ix, iy, iz) the integer coordinates of the cell at its
 *                         depth; unit coordinate u = (word >> 8) * 2^-24 in f32 and the point min + (max - min) * u in f32
 *                         like Eigen's AlignedBox::sample(), cast to f64 for FApprox (Octree.cpp:1222, 1242). A weight
 *                         then depends only on (seed, cell, degree, coefficients), never on the schedule. */
static int      g_nearnessMc = 0;
static uint64_t g_nearnessSeed = 0;
void hporacle_set_nearness_mc(int on, uint64_t seed) { g_nearnessMc = on; g_nearnessSeed = seed; }

static void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1)
{
    for (int r = 0; r < 10; ++r)
    {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
        c[0] = n0; c[1] = (uint32_t)p1; c[2] = n2; c[3] = (uint32_t)p0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}

/* test hook: one Philox4x32-10 block (tests/test_oracle_vs_ref.py checks it against the Random123 known-answer vectors) */
void hporacle_philox(uint32_t c[4], uint32_t k0, uint32_t k1) { philox4x32_10(c, k0, k1); }

static double f_approx(const double* coeffs, uint32_t degree, const Box* aabb, const double pt[3], uint32_t depth);

static double nearness_mean(const double* coeffs, uint32_t degree, const Box* aabb, uint32_t depth)
{
    if (!g_nearnessMc)
    {
        const double nl = NL[0][depth];
        return fabs(coeffs[0] * (nl * nl * nl));
    }
    uint32_t cell[3];
    for (int a = 0; a < 3; ++a) cell[a] = (uint32_t)((aabb->mn[a] + 0.5f) * (float)(1u << depth));      /* dyadic cells of [-0.5, 0.5]^3: exact */
    double sum = 0.0;
    for (uint32_t s = 0; s < 100; ++s)                                                                  /* nSamples, Octree.cpp:1216, 1236 */
    {
        uint32_t c[4] = { cell[0], cell[1], cell[2], depth | (degree << 8) | (s << 16) };
        philox4x32_10(c, (uint32_t)g_nearnessSeed, (uint32_t)(g_nearnessSeed >> 32));
        double pt[3];
        for (int a = 0; a < 3; ++a)
        {
            const float u = (float)(c[a] >> 8) * 0x1p-24f;
            const float ext = aabb->mx[a] - aabb->mn[a];
            const float x = aabb->mn[a] + ext * u;
            pt[a] = (double)x;
        }
        sum += f_approx(coeffs, degree, aabb, pt, depth);
    }
    sum /= 100;
    return fabs(sum);
}

static double nearness_weight(const hpsdf_config* cfg, const double* coeffs, uint32_t degree, const Box* aabb, uint32_t depth)
{
    if (cfg->nearness_type == HPSDF_NEARNESS_NONE) return 1.0;
    const double m = nearness_mean(coeffs, degree, aabb, depth);
    const double d = sqrt(3.0);
    if (cfg->nearness_type == HPSDF_NEARNESS_POLYNOMIAL)
    {
        const double k = pow(1.0 - m / d, cfg->nearness_strength);
        const double lo = (k < 0.0) ? 0.0 : k;      /* std::max(k, 0.0) */
        return (lo < 1.0) ? lo : 1.0;               /* std::min(1.0, lo) */
    }
    return exp(-1.0 * cfg->nearness_strength * m / d);
}

static void log_apply(Tree* t, ApplyRecord r)
{
    if (t->nLog == t->capLog) { t->capLog = t->capLog ? 2 * t->capLog : 8192; t->log = (ApplyRecord*)realloc(t->log, t->capLog * sizeof(ApplyRecord)); }
    t->log[t->nLog++] = r;
}

/* RunBuildThreadPool + TickBuildThread (Octree.cpp:194-309, 558-659) as the deterministic strict-greedy schedule. */
static void greedy_build(Tree* t, uint32_t maxDegree, uint32_t maxDepth, uint32_t totalMode, int threads)
{
    double total = pow(8, 4) * INITIAL_NODE_ERR;      /* Octree.cpp:212 */
    long double exactSum = 0.0L;
    long unfitted = (long)t->nHeap;
    const double thr = t->cfg.target_error_threshold;
    (void)threads;

    for (;;)
    {
        const double check = totalMode == HPSDF_TOTAL_EXACT_SUM ? (unfitted > 0 ? INFINITY : (double)exactSum) : total;
        if (check < thr || t->nHeap == 0) break;                                       /* Octree.cpp:216 */

        const HeapItem top = heap_pop(t);                                              /* Octree.cpp:231-232 */
        const Node node = t->nodes[top.idx];
        const double err = top.err;
        const int isCoarse = fabs(err - INITIAL_NODE_ERR) < DBL_EPSILON;               /* Octree.cpp:806, 831 */
        const uint32_t p = node.degree, depth = node.depth;
        const int doH = !isCoarse && depth < maxDepth;
        const int doP = isCoarse || p < maxDegree;

        double* hC[8] = { 0 }; double* pC = NULL;
        double rawH[8] = { 0 }, rawP = 0.0, hErr[8] = { 0 }, pErr = 0.0, hImp = 0.0, pImp = 0.0;
        Box childBox[8];
        if (doH) for (uint32_t i = 0; i < 8; ++i) { hC[i] = (double*)malloc(sizeof(double) * COUNT[p]); childBox[i] = corner_aabb(&node.aabb, i); }
        if (doP)
        {
            pC = (double*)malloc(sizeof(double) * COUNT[isCoarse ? 2 : p + 1]);
            if (!isCoarse) memcpy(pC, node.coeffs, sizeof(double) * COUNT[p]);          /* Octree.cpp:846-848 */
        }
        #pragma omp parallel for schedule(dynamic, 1) num_threads(threads) if (threads > 1)
        for (int f = 0; f < 9; ++f)
        {
            if (f < 8) { if (doH) rawH[f] = fit_polynomial(t, hC[f], 0, &childBox[f], p, depth + 1); }                 /* Octree.cpp:820 */
            else if (doP) rawP = isCoarse ? fit_polynomial(t, pC, 0, &node.aabb, 2, depth)                             /* Octree.cpp:840 */
                                          : fit_polynomial(t, pC, p, &node.aabb, p + 1, depth);                        /* Octree.cpp:851 */
        }
        t->jobs++;
        if (doH)
        {
            double maxNew = 0.0;
            for (uint32_t i = 0; i < 8; ++i) { hErr[i] = rawH[i] * nearness_weight(&t->cfg, hC[i], p, &childBox[i], depth + 1); maxNew = (maxNew < hErr[i]) ? hErr[i] : maxNew; }
            hImp = (1.0 / (7.0 * COUNT[p])) * (err - 8.0 * maxNew);                                                    /* Octree.cpp:825 */
            t->fits += 8;
        }
        if (doP)
        {
            pErr = rawP * nearness_weight(&t->cfg, pC, isCoarse ? 2u : p + 1u, &node.aabb, depth);
            pImp = isCoarse ? pErr : (1.0 / (COUNT[p + 1] - COUNT[p])) * (err - 8.0 * pErr);                           /* Octree.cpp:842, 854 */
            t->fits += 1;
        }
        /* Octree.cpp:600-601 (BASIS_MAX_DEGREE-1 -> maxDegree, TREE_MAX_DEPTH -> maxDepth); a coarse cell always takes
         * its degree-2 fit (the reference is undefined if that fit's error is exactly 0, SURVEY.md App. C). */
        const int refineP = isCoarse || (p < maxDegree && (depth == maxDepth || pImp > hImp));
        const int refineH = depth < maxDepth && !refineP;

        ApplyRecord rec = { top.idx, 0u, p, err, 0.0, pImp, hImp, 0.0 };
        if (refineP)
        {
            for (int i = 0; i < 8; ++i) free(hC[i]);
            free(t->nodes[top.idx].coeffs);
            total += (pErr - err);                                                     /* Octree.cpp:257 */
            if (isCoarse) unfitted--; else exactSum -= (long double)err;
            exactSum += (long double)pErr;
            t->nodes[top.idx].coeffs = pC;                                             /* Octree.cpp:286 */
            t->nodes[top.idx].degree = (uint8_t)(isCoarse ? 2 : p + 1);
            heap_push(t, top.idx, pErr);                                               /* Octree.cpp:289-290 */
            t->appliedP++;
            rec.kind = 0; rec.newErr = pErr;
        }
        else if (refineH)
        {
            free(pC);
            free(t->nodes[top.idx].coeffs);                                            /* Octree.cpp:265-272 */
            t->nodes[top.idx].coeffs = NULL;
            t->nodes[top.idx].degree = INTERNAL_TAG;
            subdivide(t, top.idx);
            total -= err;
            exactSum -= (long double)err;
            double mx = 0.0;
            for (uint32_t i = 0; i < 8; ++i)
            {
                const uint64_t c = t->nodes[top.idx].child + i;                        /* Octree.cpp:275-290 */
                total += hErr[i];
                exactSum += (long double)hErr[i];
                t->nodes[c].coeffs = hC[i];
                t->nodes[c].degree = (uint8_t)p;
                heap_push(t, c, hErr[i]);
                mx = mx < hErr[i] ? hErr[i] : mx;
            }
            t->appliedH++;
            rec.kind = 1; rec.newErr = mx;
        }
        else
        {
            for (int i = 0; i < 8; ++i) free(hC[i]);                                   /* Octree.cpp:643-655 */
            free(pC);
            continue;
        }
        rec.totalAfter = totalMode == HPSDF_TOTAL_EXACT_SUM ? (unfitted > 0 ? INFINITY : (double)exactSum) : total;
        log_apply(t, rec);
    }
    t->finalTotal = totalMode == HPSDF_TOTAL_EXACT_SUM ? (double)exactSum : total;
}

/* ReallocCoeffs, Octree.cpp:474-555: DFS from the root by child slot, leaves packed in visiting order. */
static void pack_dfs(Tree* t, uint64_t idx, size_t* cur)
{
    Node* n = &t->nodes[idx];
    if (n->child == NO_CHILD)
    {
        memcpy(t->store + *cur, n->coeffs, sizeof(double) * COUNT[n->degree]);
        free(n->coeffs); n->coeffs = NULL;
        n->cstart = *cur; *cur += COUNT[n->degree];
    }
    else for (uint32_t i = 0; i < 8; ++i) pack_dfs(t, t->nodes[idx].child + i, cur);
}

static void realloc_coeffs(Tree* t)
{
    size_t n = 0;
    for (size_t i = 0; i < t->nNodes; ++i) if (t->nodes[i].degree != INTERNAL_TAG) n += COUNT[t->nodes[i].degree];
    t->store = (double*)malloc(sizeof(double) * (n ? n : 1));
    t->nCoeffs = n;
    size_t cur = 0;
    for (uint32_t i = 0; i < 8; ++i) pack_dfs(t, t->nodes[0].child + i, &cur);       /* the traveller starts at the root's children */
}

/* ---- Query ----------------------------------------------------------------------------------------------- */
/* FApprox, Octree.cpp:859-901 */
static double f_approx(const double* coeffs, uint32_t degree, const Box* aabb, const double pt[3], uint32_t depth)
{
    float cf[3];
    box_center(aabb, cf);
    const double scale = (double)(2 << depth);
    double lut[MAXDEG + 1][3];
    for (int i = 0; i < 3; ++i)
    {
        const double u = (pt[i] - (double)cf[i]) * scale;
        lut[0][i] = NL[0][depth];
        double m2 = 0.0, m1 = 1.0, l = 1.0;
        for (uint32_t j = 1; j <= degree; ++j)
        {
            l = REC[j][0] * u * m1 - REC[j][1] * m2; m2 = m1; m1 = l;
            lut[j][i] = l * NL[j][depth];
        }
    }
    double f = 0.0;
    for (uint32_t i = 0; i < COUNT[degree]; ++i)
    {
        double lp = 1.0;
        for (int j = 0; j < 3; ++j) lp *= lut[BIDX[i][j]][j];
        f += coeffs[i] * lp;
    }
    return f;
}

/* descent shared by Query / QueryWithGradient, Octree.cpp:662-702 */
static int64_t find_leaf(const Tree* t, const double x[3], double pt[3])
{
    for (int i = 0; i < 3; ++i) pt[i] = (x[i] - t->rootCentre[i]) * t->rootInvSizes[i];
    const Box* r = &t->nodes[0].aabb;
    for (int i = 0; i < 3; ++i) { const float f = (float)pt[i]; if (!(r->mn[i] <= f && f <= r->mx[i])) return -1; }
    uint64_t cur = 0;
    for (;;)
    {
        const Box* b = &t->nodes[cur].aabb;
        const float half = (b->mx[0] - b->mn[0]) * 0.5f;
        const uint64_t xi = pt[0] >= (double)(b->mn[0] + half);
        const uint64_t yi = (uint64_t)(pt[1] >= (double)(b->mn[1] + half)) << 1;
        const uint64_t zi = (uint64_t)(pt[2] >= (double)(b->mn[2] + half)) << 2;
        const uint64_t c = t->nodes[cur].child + xi + yi + zi;
        if (t->nodes[c].degree != INTERNAL_TAG) return (int64_t)c;
        cur = c;
    }
}

static double query_one(const Tree* t, const double x[3])
{
    double pt[3];
    const int64_t leaf = find_leaf(t, x, pt);
    if (leaf < 0) return DBL_MAX;                                                     /* Octree.cpp:668-671 */
    const Node* n = &t->nodes[leaf];
    return f_approx(t->store + n->cstart, n->degree, &n->aabb, pt, n->depth);
}

/* FApproxWithGradient, Octree.cpp:904-985 */
static double query_gradient_one(const Tree* t, const double x[3], double g[3])
{
    double pt[3];
    const int64_t leaf = find_leaf(t, x, pt);
    if (leaf < 0) return DBL_MAX;
    const Node* n = &t->nodes[leaf];
    const double* coeffs = t->store + n->cstart;
    const uint32_t degree = n->degree, depth = n->depth;
    float cf[3];
    box_center(&n->aabb, cf);
    const double scale = (double)(2 << depth), eps = 0.0001;
    double lut[MAXDEG + 1][3][3];
    for (int i = 0; i < 3; ++i)
    {
        const double u = (pt[i] - (double)cf[i]) * scale;
        const double us[3] = { u, u + eps, u - eps };
        for (int v = 0; v < 3; ++v)
        {
            lut[0][i][v] = NL[0][depth];
            double m2 = 0.0, m1 = 1.0, l = 1.0;
            for (uint32_t j = 1; j <= degree; ++j)
            {
                l = REC[j][0] * us[v] * m1 - REC[j][1] * m2; m2 = m1; m1 = l;
                lut[j][i][v] = l * NL[j][depth];
            }
        }
    }
    for (int k = 0; k < 3; ++k)
    {
        double fp = 0.0, fm = 0.0;
        for (uint32_t i = 0; i < COUNT[degree]; ++i) { fp += coeffs[i] * lut[BIDX[i][k]][k][1]; fm += coeffs[i] * lut[BIDX[i][k]][k][2]; }
        g[k] = (fp - fm) / (2.0 * eps);
    }
    const double nrm = sqrt(g[0] * g[0] + (g[1] * g[1] + g[2] * g[2]));
    if (nrm > 0.0) for (int k = 0; k < 3; ++k) g[k] /= nrm;
    double f = 0.0;
    for (uint32_t i = 0; i < COUNT[degree]; ++i)
    {
        double lp = 1.0;
        for (int j = 0; j < 3; ++j) lp *= lut[BIDX[i][j]][j][0];
        f += coeffs[i] * lp;
    }
    return f;
}

/* ---- continuity ------------------------------------------------------------------------------------------ */
typedef struct { int32_t r, c; double v; } Trip;
typedef struct { Trip* d; size_t n, cap; } TripVec;
typedef struct { uint64_t a, b; uint8_t dim; } FaceJob;
typedef struct { FaceJob* d; size_t n, cap; } JobVec;

static void trip_push(TripVec* v, uint64_t r, uint64_t c, double x)
{
    if (v->n == v->cap) { v->cap = v->cap ? 2 * v->cap : (1u << 20); v->d = (Trip*)realloc(v->d, v->cap * sizeof(Trip)); }
    v->d[v->n].r = (int32_t)r; v->d[v->n].c = (int32_t)c; v->d[v->n].v = x; v->n++;
}

static void job_push(JobVec* v, uint64_t a, uint64_t b, uint8_t dim)
{
    if (v->n == v->cap) { v->cap = v->cap ? 2 * v->cap : 65536; v->d = (FaceJob*)realloc(v->d, v->cap * sizeof(FaceJob)); }
    v->d[v->n].a = a; v->d[v->n].b = b; v->d[v->n].dim = dim; v->n++;
}

/* FaceProc, Octree.cpp:1574-1612. NodeProc is run from the root only: the reference runs it from every node and lets
 * procMap drop the repeats (Octree.cpp:1675-1678); a face reached from the root is reached exactly once. */
static void face_proc(const Tree* t, uint64_t a, uint64_t b, uint8_t dim, JobVec* jobs)
{
    const int ac = t->nodes[a].child != NO_CHILD, bc = t->nodes[b].child != NO_CHILD;
    if (ac || bc)
    {
        for (uint32_t i = 0; i < 4; ++i)
            face_proc(t, ac ? t->nodes[a].child + FACE[dim][i][1] : a, bc ? t->nodes[b].child + FACE[dim][i][0] : b, dim, jobs);
    }
    else
    {
        const int aLow = t->nodes[a].aabb.mn[dim] < t->nodes[b].aabb.mn[dim];
        job_push(jobs, aLow ? a : b, aLow ? b : a, dim);
    }
}

/* NodeProc, Octree.cpp:1549-1571 */
static void node_proc(const Tree* t, uint64_t idx, JobVec* jobs)
{
    const Node* n = &t->nodes[idx];
    if (n->child == NO_CHILD) return;
    for (uint32_t i = 0; i < 8; ++i) node_proc(t, n->child + i, jobs);
    for (uint8_t d = 0; d < 3; ++d)
        for (uint32_t j = 0; j < 4; ++j) face_proc(t, n->child + FACE[d][j][0], n->child + FACE[d][j][1], d, jobs);
}

/* EvaluateSharedFaceIntegralAnalytically, Octree.cpp:1459-1546 */
static void face_analytic(const Tree* t, uint64_t ia, uint64_t ib, uint8_t dim, TripVec* out)
{
    const Node* A = &t->nodes[ia]; const Node* B = &t->nodes[ib];
    const uint32_t t1 = (dim + 1) % 3, t2 = (dim + 2) % 3;
    const uint32_t nA = COUNT[A->degree], nB = COUNT[B->degree];
    for (uint32_t i = 0; i < nA; ++i) for (uint32_t j = 0; j < nA; ++j)
    {
        if (BIDX[i][t1] != BIDX[j][t1] || BIDX[i][t2] != BIDX[j][t2]) continue;
        double v = 1.0;
        v *= LpX(BIDX[i][dim], 1.0); v *= NL[BIDX[i][dim]][A->depth]; v *= LpX(BIDX[j][dim], 1.0); v *= NL[BIDX[j][dim]][A->depth];
        trip_push(out, A->cstart + i, A->cstart + j, v);
    }
    for (uint32_t i = 0; i < nA; ++i) for (uint32_t j = 0; j < nB; ++j)
    {
        if (BIDX[i][t1] != BIDX[j][t1] || BIDX[i][t2] != BIDX[j][t2]) continue;
        double v = -1.0;
        v *= LpX(BIDX[i][dim], 1.0); v *= NL[BIDX[i][dim]][A->depth]; v *= LpX(BIDX[j][dim], -1.0); v *= NL[BIDX[j][dim]][B->depth];
        trip_push(out, A->cstart + i, B->cstart + j, v);
        trip_push(out, B->cstart + j, A->cstart + i, v);
    }
    for (uint32_t i = 0; i < nB; ++i) for (uint32_t j = 0; j < nB; ++j)
    {
        if (BIDX[i][t1] != BIDX[j][t1] || BIDX[i][t2] != BIDX[j][t2]) continue;
        double v = 1.0;
        v *= LpX(BIDX[i][dim], -1.0); v *= NL[BIDX[i][dim]][B->depth]; v *= LpX(BIDX[j][dim], -1.0); v *= NL[BIDX[j][dim]][B->depth];
        trip_push(out, B->cstart + i, B->cstart + j, v);
    }
}

/* EvaluateSharedFaceIntegralNumerically, Octree.cpp:1250-1456 */
static void face_numeric(const Tree* t, uint64_t ia, uint64_t ib, uint8_t dim, TripVec* out)
{
    const Node* A = &t->nodes[ia]; const Node* B = &t->nodes[ib];
    const uint32_t t1 = (dim + 1) % 3, t2 = (dim + 2) % 3;
    /* shared face = A.aabb clamped to B.aabb (intersection), Octree.cpp:1265-1267 */
    double faceScale[3];
    for (int i = 0; i < 3; ++i)
    {
        const float lo = A->aabb.mn[i] > B->aabb.mn[i] ? A->aabb.mn[i] : B->aabb.mn[i];
        const float hi = A->aabb.mx[i] < B->aabb.mx[i] ? A->aabb.mx[i] : B->aabb.mx[i];
        faceScale[i] = (double)(hi - lo) * 0.5;
    }
    const uint32_t maxDeg = A->degree > B->degree ? A->degree : B->degree;
    const uint32_t gq = maxDeg * (maxDeg + 1) / 2, n = maxDeg + 1;                      /* SumToN[maxDegree] .. SumToN[maxDegree+1] */
    const uint32_t depthDiff = A->depth > B->depth ? (uint32_t)(A->depth - B->depth) : (uint32_t)(B->depth - A->depth);
    const double invDist = 1.0 / pow(2.0, (double)depthDiff);
    double invTr[3] = { 0.0, 0.0, 0.0 };
    float ca[3], cb[3];
    box_center(&A->aabb, ca); box_center(&B->aabb, cb);
    if (A->depth > B->depth)
    {   /* f32 arithmetic until the division by (sizes * 0.5), which promotes to f64 (Octree.cpp:1282-1283) */
        invTr[t1] = (double)(ca[t1] - cb[t1]) / ((double)(A->aabb.mx[t1] - A->aabb.mn[t1]) * 0.5);
        invTr[t2] = (double)(ca[t2] - cb[t2]) / ((double)(A->aabb.mx[t2] - A->aabb.mn[t2]) * 0.5);
    }
    else
    {
        invTr[t1] = (double)(cb[t1] - ca[t1]) / ((double)(B->aabb.mx[t1] - B->aabb.mn[t1]) * 0.5);
        invTr[t2] = (double)(cb[t2] - ca[t2]) / ((double)(B->aabb.mx[t2] - B->aabb.mn[t2]) * 0.5);
    }
    for (int i = 0; i < 3; ++i) invTr[i] *= invDist;

    const uint32_t nA = COUNT[A->degree], nB = COUNT[B->degree];
    for (int block = 0; block < 3; ++block)       /* 0: AA, 1: AB (+BA), 2: BB */
    {
        const Node* R = block == 2 ? B : A; const Node* Cn = block == 0 ? A : B;
        const uint32_t nR = block == 2 ? nB : nA, nC = block == 0 ? nA : nB;
        for (uint32_t i = 0; i < nR; ++i) for (uint32_t j = 0; j < nC; ++j)
        {
            double integral = 0.0;
            for (uint32_t x = 0; x < n; ++x) for (uint32_t y = 0; y < n; ++y)
            {
                double a[3], b[3];
                a[dim] = 1.0;  a[t1] = ROOTS[gq + x]; a[t2] = ROOTS[gq + y];
                b[dim] = -1.0; b[t1] = ROOTS[gq + x]; b[t2] = ROOTS[gq + y];
                if (B->depth > A->depth) { a[t1] = a[t1] * invDist + invTr[t1]; a[t2] = a[t2] * invDist + invTr[t2]; }
                else if (A->depth > B->depth) { b[t1] = b[t1] * invDist + invTr[t1]; b[t2] = b[t2] * invDist + invTr[t2]; }
                const double* sr = block == 2 ? b : a;      /* sample seen by the row function */
                const double* sc = block == 0 ? a : b;      /* sample seen by the column function */
                double area = WEIGHTS[gq + x] * WEIGHTS[gq + y];
                for (uint32_t k = 0; k < 3; ++k) { area *= LpX(BIDX[i][k], sr[k]); area *= LpX(BIDX[j][k], sc[k]); }
                integral += area;
            }
            double bw = 1.0;
            for (uint32_t k = 0; k < 3; ++k) { bw *= NL[BIDX[i][k]][R->depth]; bw *= NL[BIDX[j][k]][Cn->depth]; }
            if (block == 1) integral *= faceScale[t1] * faceScale[t2] * bw * -1.0;
            else            integral *= faceScale[t1] * faceScale[t2] * bw;
            if (fabsf((float)integral) > 0.000001f)                                       /* EPSILON_F32, Literals.h:13 */
            {
                trip_push(out, R->cstart + i, Cn->cstart + j, integral);
                if (block == 1) trip_push(out, Cn->cstart + j, R->cstart + i, integral);
            }
        }
    }
}

static int trip_cmp(const void* a, const void* b)
{
    const Trip* x = (const Trip*)a; const Trip* y = (const Trip*)b;
    if (x->r != y->r) return x->r < y->r ? -1 : 1;
    if (x->c != y->c) return x->c < y->c ? -1 : 1;
    return 0;
}

typedef struct { size_t n; int64_t* rowPtr; int32_t* col; double* val; } Csr;

/* RunContinuityThreadPool + the lambda diagonal + setFromTriplets, Octree.cpp:1663-1735 */
static Csr assemble_continuity(const Tree* t, int withDiagonal)
{
    JobVec jobs = { 0 };
    node_proc(t, 0, &jobs);
    TripVec tr = { 0 };
    for (size_t i = 0; i < jobs.n; ++i)
    {
        const FaceJob* j = &jobs.d[i];
        if (t->nodes[j->a].depth == t->nodes[j->b].depth) face_analytic(t, j->a, j->b, j->dim, &tr);    /* Octree.cpp:1651-1658 */
        else face_numeric(t, j->a, j->b, j->dim, &tr);
    }
    free(jobs.d);
    if (withDiagonal) for (size_t i = 0; i < t->nCoeffs; ++i) trip_push(&tr, i, i, t->cfg.continuity_strength);        /* Octree.cpp:1724-1729 */
    qsort(tr.d, tr.n, sizeof(Trip), trip_cmp);     /* order of equal (r,c) entries only changes the last ulp of the sum */
    Csr m; m.n = t->nCoeffs;
    m.rowPtr = (int64_t*)calloc(m.n + 1, sizeof(int64_t));
    m.col = (int32_t*)malloc(sizeof(int32_t) * (tr.n ? tr.n : 1)); m.val = (double*)malloc(sizeof(double) * (tr.n ? tr.n : 1));
    size_t nnz = 0;
    for (size_t i = 0; i < tr.n; ++i)
    {
        if (nnz > 0 && i > 0 && tr.d[i].r == tr.d[i - 1].r && tr.d[i].c == tr.d[i - 1].c) { m.val[nnz - 1] += tr.d[i].v; continue; }
        m.col[nnz] = tr.d[i].c; m.val[nnz] = tr.d[i].v; nnz++;
        m.rowPtr[tr.d[i].r + 1] = (int64_t)nnz;
    }
    for (size_t r = 0; r < m.n; ++r) if (m.rowPtr[r + 1] < m.rowPtr[r]) m.rowPtr[r + 1] = m.rowPtr[r];
    free(tr.d);
    return m;
}

static void csr_mul(const Csr* m, const double* x, double* y, int threads)
{
    (void)threads;
    #pragma omp parallel for schedule(static) num_threads(threads) if (threads > 1)
    for (long r = 0; r < (long)m->n; ++r)
    {
        double s = 0.0;
        for (int64_t k = m->rowPtr[r]; k < m->rowPtr[r + 1]; ++k) s += m->val[k] * x[m->col[k]];
        y[r] = s;
    }
}

static double dotn(const double* a, const double* b, size_t n) { double s = 0.0; for (size_t i = 0; i < n; ++i) s += a[i] * b[i]; return s; }

/* PerformContinuityPostProcess, Octree.cpp:1717-1762: (M + lambda I) x = lambda c, x0 = lambda c, CG with Eigen's loop and
 * stopping rule |r|^2 < tol^2 |b|^2 (max 2n iterations); diagonal preconditioner (Eigen's IC is not restated: unpinned). */
static void continuity_post_process(Tree* t, double tol, int threads)
{
    const size_t n = t->nCoeffs;
    Csr m = assemble_continuity(t, 1);
    double* b = (double*)malloc(sizeof(double) * n); double* x = (double*)malloc(sizeof(double) * n);
    double* r = (double*)malloc(sizeof(double) * n); double* p = (double*)malloc(sizeof(double) * n);
    double* z = (double*)malloc(sizeof(double) * n); double* tmp = (double*)malloc(sizeof(double) * n);
    double* invDiag = (double*)malloc(sizeof(double) * n);
    for (size_t i = 0; i < n; ++i)
    {
        b[i] = t->store[i] * t->cfg.continuity_strength; x[i] = b[i]; invDiag[i] = 1.0;
        for (int64_t k = m.rowPtr[i]; k < m.rowPtr[i + 1]; ++k) if ((size_t)m.col[k] == i && m.val[k] != 0.0) invDiag[i] = 1.0 / m.val[k];
    }
    csr_mul(&m, x, tmp, threads);
    for (size_t i = 0; i < n; ++i) r[i] = b[i] - tmp[i];
    const double rhs2 = dotn(b, b, n);
    const double threshold = fmax(tol * tol * rhs2, DBL_MIN);
    double res2 = dotn(r, r, n);
    uint64_t it = 0;
    if (rhs2 > 0.0 && res2 >= threshold)
    {
        for (size_t i = 0; i < n; ++i) p[i] = invDiag[i] * r[i];
        double absNew = dotn(r, p, n);
        while (it < 2 * n)
        {
            csr_mul(&m, p, tmp, threads);
            const double alpha = absNew / dotn(p, tmp, n);
            for (size_t i = 0; i < n; ++i) { x[i] += alpha * p[i]; r[i] -= alpha * tmp[i]; }
            res2 = dotn(r, r, n);
            if (res2 < threshold) break;
            for (size_t i = 0; i < n; ++i) z[i] = invDiag[i] * r[i];
            const double absOld = absNew;
            absNew = dotn(r, z, n);
            const double beta = absNew / absOld;
            for (size_t i = 0; i < n; ++i) p[i] = z[i] + beta * p[i];
            it++;
        }
    }
    t->cgIterations = it;
    t->cgError = rhs2 > 0.0 ? sqrt(res2 / rhs2) : 0.0;
    memcpy(t->store, x, sizeof(double) * n);                                          /* Octree.cpp:1756 */
    free(b); free(x); free(r); free(p); free(z); free(tmp); free(invDiag); free(m.rowPtr); free(m.col); free(m.val);
}

/* MESH primitives of a program: handle = OMesh* (hporacle_mesh_create); the f64 point is cast to f32 and the f32 distance
 * widened, the glue the reference implies (Include/Meshing/Mesh.h:53-54). OCTREE primitives: handle = Tree*. */
static double query_one(const Tree* t, const double x[3]);
static double builtin_ext(uint32_t op, const void* handle, const double x[3])
{
    if (op == HPSDF_PRIM_MESH)
    {
        const mv3 p = { (float)x[0], (float)x[1], (float)x[2] };
        return (double)omesh_signed_distance((const OMesh*)handle, p, 1);
    }
    if (op == HPSDF_PRIM_OCTREE) return query_one((const Tree*)handle, x);
    return NAN;
}

void* hporacle_mesh_create(const float* verts, size_t nv, const uint32_t* tris, size_t nt) { return omesh_create(verts, nv, tris, nt); }
void  hporacle_mesh_destroy(void* m) { omesh_free((OMesh*)m); }
/* The half-edge twins of a created mesh, 3 per triangle (for tests of the pairing rule). */
void  hporacle_mesh_half_edges(const void* m, uint32_t* out) { memcpy(out, ((const OMesh*)m)->he, 3 * ((const OMesh*)m)->nt * 4); }
void  hporacle_mesh_sdf(void* m, const float* xyz, size_t n, float* out, int useBvh, int threads)
{
    (void)threads;
    #pragma omp parallel for schedule(dynamic, 64) num_threads(threads) if (threads > 1)
    for (long i = 0; i < (long)n; ++i)
    {
        const mv3 p = { xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2] };
        out[i] = omesh_signed_distance((const OMesh*)m, p, useBvh);
    }
}

/* ---- public entry points (ctypes) ------------------------------------------------------------------------ */
static double now_s(void) { struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec + 1e-9 * ts.tv_nsec; }

static Tree* tree_new(const hpsdf_config* cfg, const hpsdf_sdf_instr* prog, uint32_t n, hporacle_ext_eval ext)
{
    hporacle_init();
    Tree* t = (Tree*)calloc(1, sizeof(Tree));
    t->cfg = *cfg;
    if (n) { t->prog = (hpsdf_sdf_instr*)malloc(sizeof(hpsdf_sdf_instr) * n); memcpy(t->prog, prog, sizeof(hpsdf_sdf_instr) * n); }
    t->nprog = n; t->ext = ext ? ext : builtin_ext;
    set_root_mapping(t);
    return t;
}

/* Octree::Create, Octree.cpp:312-352, deterministic schedule. cgTol <= 0 selects the reference's (double)1e-6f. */
void* hporacle_build(const hpsdf_config* cfg, const hpsdf_sdf_instr* prog, uint32_t n, uint32_t maxDegree, uint32_t maxDepth,
                     uint32_t totalMode, double cgTol, int threads, hporacle_ext_eval ext)
{
    Tree* t = tree_new(cfg, prog, n, ext);
    if (threads < 1) threads = 1;
    const double t0 = now_s();
    create_root_and_coarse_grid(t);
    greedy_build(t, maxDegree, maxDepth, totalMode, threads);
    const double t1 = now_s();
    realloc_coeffs(t);
    if (cfg->continuity_enforce) continuity_post_process(t, cgTol > 0.0 ? cgTol : (double)0.000001f, threads);
    const double t2 = now_s();
    t->seconds = t2 - t0; t->continuitySeconds = t2 - t1;
    return t;
}

void hporacle_destroy(void* h)
{
    Tree* t = (Tree*)h;
    if (!t) return;
    for (size_t i = 0; i < t->nNodes; ++i) free(t->nodes[i].coeffs);
    free(t->nodes); free(t->store); free(t->heap); free(t->log); free(t->prog); free(t);
}

/* ToMemoryBlock, Octree.cpp:424-456; LP64 offsets per SURVEY.md App. B */
size_t hporacle_block_size(void* h) { Tree* t = (Tree*)h; return 8 + 8 * t->nCoeffs + 8 + 56 * t->nNodes + 80; }

void hporacle_block_copy(void* h, void* dst)
{
    Tree* t = (Tree*)h;
    uint8_t* p = (uint8_t*)dst;
    memset(p, 0, hporacle_block_size(h));
    const uint64_t nc = t->nCoeffs, nn = t->nNodes;
    memcpy(p, &nc, 8); p += 8;
    memcpy(p, t->store, 8 * nc); p += 8 * nc;
    memcpy(p, &nn, 8); p += 8;
    for (size_t i = 0; i < t->nNodes; ++i, p += 56)
    {
        const Node* n = &t->nodes[i];
        memcpy(p + 0, &n->child, 8); memcpy(p + 8, n->aabb.mn, 12); memcpy(p + 20, n->aabb.mx, 12);
        memcpy(p + 32, &n->cstart, 8); p[40] = n->degree; p[48] = n->depth;
    }
    memcpy(p, &t->cfg, 80);
}

/* FromMemoryBlock, Octree.cpp:403-421 */
void* hporacle_from_block(const void* ptr, size_t size)
{
    const uint8_t* p = (const uint8_t*)ptr;
    uint64_t nc, nn;
    memcpy(&nc, p, 8);
    memcpy(&nn, p + 8 + 8 * nc, 8);
    if (size != 8 + 8 * nc + 8 + 56 * nn + 80) return NULL;
    hpsdf_config cfg;
    memcpy(&cfg, p + 16 + 8 * nc + 56 * nn, 80);
    Tree* t = tree_new(&cfg, NULL, 0, NULL);
    t->nCoeffs = nc; t->store = (double*)malloc(8 * (nc ? nc : 1)); memcpy(t->store, p + 8, 8 * nc);
    const uint8_t* q = p + 16 + 8 * nc;
    for (uint64_t i = 0; i < nn; ++i, q += 56)
    {
        const uint64_t k = push_node(t);
        Node* n = &t->nodes[k];
        memcpy(&n->child, q, 8); memcpy(n->aabb.mn, q + 8, 12); memcpy(n->aabb.mx, q + 20, 12);
        memcpy(&n->cstart, q + 32, 8); n->degree = q[40]; n->depth = q[48];
    }
    return t;
}

void hporacle_query(void* h, const double* xyz, size_t n, double* out, int threads)
{
    const Tree* t = (const Tree*)h;
    (void)threads;
    #pragma omp parallel for schedule(static) num_threads(threads) if (threads > 1)
    for (long i = 0; i < (long)n; ++i) out[i] = query_one(t, xyz + 3 * i);
}

/* Octree::QueryRay (Octree.cpp:705-746) with Ray::Ray (Ray.cpp:5-14) and Ray::IntersectAABB (Ray.cpp:17-65), statement by
 * statement: the origin is mapped into the unit cube, the direction is not (:713); outside the root the march starts from the
 * a_ output of IntersectAABB (entry parameter in x, slab parameters in y and z) (:715-719); samples go through Query (:729). */
void hporacle_query_ray(void* h, const double* origins, const double* dirs, size_t n, double tMax, unsigned char* hit, double* tOut)
{
    const Tree* t = (const Tree*)h;
    for (size_t r = 0; r < n; ++r)
    {
        double o[3], dir[3], inv[3], intMin[3];
        int sign[3];
        for (int a = 0; a < 3; ++a)
        {
            o[a] = (origins[3 * r + a] - t->rootCentre[a]) * t->rootInvSizes[a];
            dir[a] = dirs[3 * r + a];
            inv[a] = 1.0 / dir[a];
            sign[a] = inv[a] < 0.0;
            intMin[a] = o[a];
        }
        const Box* root = &t->nodes[0].aabb;
        int inside = 1, ok = 1;
        for (int a = 0; a < 3; ++a) { const float f = (float)o[a]; if (!(root->mn[a] <= f && f <= root->mx[a])) inside = 0; }
        if (!inside)
        {
            const double bounds[2][3] = { { root->mn[0], root->mn[1], root->mn[2] }, { root->mx[0], root->mx[1], root->mx[2] } };
            double a_[3] = { o[0], o[1], o[2] }, b_[3] = { 0.0, 0.0, 0.0 };
            a_[0] = (bounds[sign[0]][0] - o[0]) * inv[0];     b_[0] = (bounds[1 - sign[0]][0] - o[0]) * inv[0];
            a_[1] = (bounds[sign[1]][1] - o[1]) * inv[1];     b_[1] = (bounds[1 - sign[1]][1] - o[1]) * inv[1];
            if ((a_[0] > b_[1]) || (a_[1] > b_[0])) ok = 0;
            if (ok)
            {
                if (a_[1] > a_[0]) a_[0] = a_[1];
                if (b_[1] < b_[0]) b_[0] = b_[1];
                a_[2] = (bounds[sign[2]][2] - o[2]) * inv[2]; b_[2] = (bounds[1 - sign[2]][2] - o[2]) * inv[2];
                if ((a_[0] > b_[2]) || (a_[2] > b_[0])) ok = 0;
                if (ok)
                {
                    if (a_[2] > a_[0]) a_[0] = a_[2];
                    intMin[0] = a_[0]; intMin[1] = a_[1]; intMin[2] = a_[2];
                }
            }
        }
        hit[r] = 0; tOut[r] = 0.0;
        if (!ok) continue;
        double d = 0.0;
        for (unsigned s = 0; s < 200; ++s)
        {
            const double p[3] = { intMin[0] + d * dir[0], intMin[1] + d * dir[1], intMin[2] + d * dir[2] };
            const double v = query_one(t, p);
            if (v < 0.0001) { tOut[r] = v; hit[r] = 1; break; }
            d += v * 0.95 + 0.0001;
            if (d > tMax) break;
        }
    }
}

void hporacle_query_gradient(void* h, const double* xyz, size_t n, double* out, double* grad, int threads)
{
    const Tree* t = (const Tree*)h;
    (void)threads;
    #pragma omp parallel for schedule(static) num_threads(threads) if (threads > 1)
    for (long i = 0; i < (long)n; ++i) out[i] = query_gradient_one(t, xyz + 3 * i, grad + 3 * i);
}

void hporacle_stats(void* h, double* out)
{
    Tree* t = (Tree*)h;
    out[0] = t->seconds; out[1] = t->continuitySeconds; out[2] = (double)t->fits; out[3] = (double)t->jobs;
    out[4] = (double)t->appliedP; out[5] = (double)t->appliedH; out[6] = t->finalTotal; out[7] = (double)t->cgIterations;
    out[8] = t->cgError; out[9] = (double)t->nLog;
}

void hporacle_apply_log(void* h, double* out)
{
    Tree* t = (Tree*)h;
    for (size_t i = 0; i < t->nLog; ++i)
    {
        const ApplyRecord* r = &t->log[i];
        double* o = out + 8 * i;
        o[0] = (double)r->node; o[1] = r->kind; o[2] = r->degree; o[3] = r->initialErr; o[4] = r->newErr; o[5] = r->pImp; o[6] = r->hImp; o[7] = r->totalAfter;
    }
}

/* One FitPolynomial, nearness None; coeffsIn (degreeIn > 0) are the kept lower shells. */
double hporacle_fit(const hpsdf_config* cfg, const hpsdf_sdf_instr* prog, uint32_t n, const float* mn, const float* mx,
                    uint32_t degreeIn, const double* coeffsIn, uint32_t degree, uint32_t depth, double* coeffsOut, hporacle_ext_eval ext)
{
    Tree* t = tree_new(cfg, prog, n, ext);
    Box b;
    memcpy(b.mn, mn, 12); memcpy(b.mx, mx, 12);
    if (degreeIn > 0) memcpy(coeffsOut, coeffsIn, sizeof(double) * COUNT[degreeIn]);
    const double e = fit_polynomial(t, coeffsOut, degreeIn, &b, degree, depth);
    hporacle_destroy(t);
    return e;
}

/* SDF program at n points in USER space (the argument of F_, Octree.cpp:327). */
void hporacle_sdf_eval_batch(const hpsdf_sdf_instr* prog, uint32_t n, const double* xyz, size_t npts, double* out, hporacle_ext_eval ext)
{
    for (size_t i = 0; i < npts; ++i) out[i] = hporacle_sdf_eval(prog, n, xyz + 3 * i, ext ? ext : builtin_ext);
}

/* Continuity matrix M (withDiagonal = 0) or M + lambda I as CSR; two-call protocol (rowPtr == NULL returns nnz). */
size_t hporacle_continuity_csr(void* h, int withDiagonal, int64_t* rowPtr, int32_t* col, double* val)
{
    Tree* t = (Tree*)h;
    Csr m = assemble_continuity(t, withDiagonal);
    const size_t nnz = (size_t)m.rowPtr[m.n];
    if (rowPtr) { memcpy(rowPtr, m.rowPtr, sizeof(int64_t) * (m.n + 1)); memcpy(col, m.col, sizeof(int32_t) * nnz); memcpy(val, m.val, sizeof(double) * nnz); }
    free(m.rowPtr); free(m.col); free(m.val);
    return nnz;
}

size_t hporacle_n_coeffs(void* h) { return ((Tree*)h)->nCoeffs; }
size_t hporacle_n_nodes(void* h) { return ((Tree*)h)->nNodes; }
