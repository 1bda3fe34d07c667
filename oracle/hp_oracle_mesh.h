/*
 * oracle/hp_oracle_mesh.h — plain-C restatement of the reference's float32 mesh signed distance.
 * TEST INFRASTRUCTURE ONLY (included by hp_oracle.c).
 *
 * Restates (file:line relative to /root/reference):
 *   Mesh::CreateHalfEdges            Source/Meshing/Mesh.cpp:87-131
 *   Mesh::SignedDistanceAtPt         Source/Meshing/Mesh.cpp:42-63
 *   Mesh::ClosestTriangleToPt        Source/Meshing/Mesh.cpp:134-159   (brute force: strict <, lowest index wins)
 *   Mesh::PseudoNormal{Face,Edge,Vertex}  Source/Meshing/Mesh.cpp:162-242
 *   ClosestSimplexToPt               Source/Meshing/Utility.cpp:5-97
 * All arithmetic is float32 in the reference's operation order (3-term sums a0 + (a1 + a2), Eigen's fixed-size
 * reduction); built with -ffp-contract=off. A median-split BVH (not the reference's NNOctree pairing, BVH.cpp:26-260 —
 * any BVH yields the same closest triangle) makes whole-octree builds affordable; `use_bvh = 0` is the brute-force loop.
 * Pinned against the reference's own Mesh (+BVH) through oracle/_ref: tests/test_oracle_vs_ref.py asserts bit equality.
 */
#ifndef HPSDF_ORACLE_MESH_H
#define HPSDF_ORACLE_MESH_H

#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <float.h>

typedef struct { float x, y, z; } mv3;
static inline mv3 mv_sub(mv3 a, mv3 b) { mv3 r = { a.x - b.x, a.y - b.y, a.z - b.z }; return r; }
static inline mv3 mv_add(mv3 a, mv3 b) { mv3 r = { a.x + b.x, a.y + b.y, a.z + b.z }; return r; }
static inline mv3 mv_mul(mv3 a, float s) { mv3 r = { a.x * s, a.y * s, a.z * s }; return r; }
static inline float mv_dot(mv3 a, mv3 b) { return a.x * b.x + (a.y * b.y + a.z * b.z); }
static inline mv3 mv_cross(mv3 a, mv3 b) { mv3 r = { a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x }; return r; }
static inline mv3 mv_normalized(mv3 a)
{
    const float z = mv_dot(a, a);
    if (z > 0.0f) { const float n = sqrtf(z); mv3 r = { a.x / n, a.y / n, a.z / n }; return r; }
    return a;
}

typedef struct { float mn[3], mx[3]; uint32_t a, b; } OBvhNode;      /* leaf: a = first slot, b = 0x80000000 | count */

typedef struct
{
    mv3*      v;   size_t nv;
    uint32_t* tri; size_t nt;
    uint32_t* he;                 /* halfEdges, 3 per triangle */
    OBvhNode* nodes; size_t nNodes, capNodes;
    uint32_t* order;              /* triangle index per BVH slot */
} OMesh;

typedef struct { int simplex, id; mv3 pt; } OClosest;                 /* simplex 0 vertex / 1 edge / 2 face */

/* ClosestSimplexToPt, Utility.cpp:5-97 */
static OClosest omesh_closest_simplex(mv3 pt, mv3 a, mv3 b, mv3 c)
{
    const float EPS = 0.000001f;
    OClosest r;
    const mv3 ab = mv_sub(b, a), ac = mv_sub(c, a), bc = mv_sub(c, b);
    const float snom = mv_dot(mv_sub(pt, a), ab), sdenom = mv_dot(mv_sub(pt, b), mv_sub(a, b));
    const float tnom = mv_dot(mv_sub(pt, a), ac), tdenom = mv_dot(mv_sub(pt, c), mv_sub(a, c));
    if (snom < EPS && tnom < EPS) { r.simplex = 0; r.id = 0; r.pt = a; return r; }
    const float unom = mv_dot(mv_sub(pt, b), bc), udenom = mv_dot(mv_sub(pt, c), mv_sub(b, c));
    if (sdenom < EPS && unom < EPS) { r.simplex = 0; r.id = 1; r.pt = b; return r; }
    if (tdenom < EPS && udenom < EPS) { r.simplex = 0; r.id = 2; r.pt = c; return r; }
    const mv3 n = mv_cross(mv_sub(b, a), mv_sub(c, a));
    const float vc = mv_dot(n, mv_cross(mv_sub(a, pt), mv_sub(b, pt)));
    if (vc < EPS && snom > EPS && sdenom > EPS) { r.simplex = 1; r.id = 0; r.pt = mv_add(a, mv_mul(ab, snom / (snom + sdenom))); return r; }
    const float va = mv_dot(n, mv_cross(mv_sub(b, pt), mv_sub(c, pt)));
    if (va < EPS && unom > EPS && udenom > EPS) { r.simplex = 1; r.id = 1; r.pt = mv_add(b, mv_mul(bc, unom / (unom + udenom))); return r; }
    const float vb = mv_dot(n, mv_cross(mv_sub(c, pt), mv_sub(a, pt)));
    if (vb < EPS && tnom > EPS && tdenom > EPS) { r.simplex = 1; r.id = 2; r.pt = mv_add(a, mv_mul(ac, tnom / (tnom + tdenom))); return r; }
    const float u = va / (va + vb + vc), v = vb / (va + vb + vc);
    const float w = 1.0f - u - v;
    r.simplex = 2; r.id = 0;
    r.pt = mv_add(mv_add(mv_mul(a, u), mv_mul(b, v)), mv_mul(c, w));
    return r;
}

static mv3 omesh_vert(const OMesh* m, uint32_t t, uint32_t k) { return m->v[m->tri[3 * t + k]]; }

/* PseudoNormalFace, Mesh.cpp:185-193 */
static mv3 omesh_face_normal(const OMesh* m, uint32_t t)
{
    return mv_normalized(mv_cross(mv_sub(omesh_vert(m, t, 1), omesh_vert(m, t, 0)), mv_sub(omesh_vert(m, t, 2), omesh_vert(m, t, 0))));
}

/* PseudoNormal, Mesh.cpp:162-242 */
static mv3 omesh_pseudo_normal(const OMesh* m, uint32_t t, int simplex, int id)
{
    if (simplex == 2) return omesh_face_normal(m, t);
    if (simplex == 1)
    {
        const uint32_t adjEdge = m->he[3 * t + (uint32_t)id], adjTri = (adjEdge - (adjEdge % 3)) / 3;
        const float PI = (float)3.14159265359;
        return mv_normalized(mv_add(mv_mul(omesh_face_normal(m, t), PI), mv_mul(omesh_face_normal(m, adjTri), PI)));
    }
    mv3 n = { 0.0f, 0.0f, 0.0f };
    uint32_t curHE = 3 * t + (uint32_t)id, curTri = t;
    size_t guard = 0;
    do
    {
        const mv3 c0 = omesh_vert(m, curTri, curHE % 3), c1 = omesh_vert(m, curTri, (curHE + 1) % 3), c2 = omesh_vert(m, curTri, (curHE + 2) % 3);
        const float ang = acosf(mv_dot(mv_normalized(mv_sub(c1, c0)), mv_normalized(mv_sub(c2, c0))));
        n = mv_add(n, mv_mul(omesh_face_normal(m, curTri), ang));
        curHE = m->he[curHE];
        curHE = ((curHE % 3) == 2) ? (curHE - 2) : (curHE + 1);
        curTri = (curHE - (curHE % 3)) / 3;
    } while (curTri != t && ++guard < 100000);
    return mv_normalized(n);
}

static float omesh_box_dist2(const OBvhNode* n, mv3 p)
{
    const float c[3] = { p.x, p.y, p.z };
    float s = 0.0f;
    for (int d = 0; d < 3; ++d)
    {
        float v = c[d];
        if (v < n->mn[d]) v = n->mn[d];
        if (v > n->mx[d]) v = n->mx[d];
        s += (v - c[d]) * (v - c[d]);
    }
    return s;
}

/* Mesh::SignedDistanceAtPt, Mesh.cpp:42-63 (brute force) / 54-63 (through a BVH) */
static float omesh_signed_distance(const OMesh* m, mv3 p, int useBvh)
{
    float best = FLT_MAX;
    uint32_t bestTri = 0xFFFFFFFFu;
    OClosest bestC;
    memset(&bestC, 0, sizeof(bestC));
    if (!useBvh || !m->nodes)
    {
        for (uint32_t t = 0; t < m->nt; ++t)                              /* Mesh.cpp:140-155: strict <, lowest index wins */
        {
            const OClosest c = omesh_closest_simplex(p, omesh_vert(m, t, 0), omesh_vert(m, t, 1), omesh_vert(m, t, 2));
            const mv3 d = mv_sub(p, c.pt);
            const float d2 = mv_dot(d, d);
            if (d2 < best) { best = d2; bestTri = t; bestC = c; }
        }
    }
    else
    {
        uint32_t stack[64];
        int sp = 0;
        stack[sp++] = 0;
        while (sp > 0)
        {
            const OBvhNode* n = &m->nodes[stack[--sp]];
            if (omesh_box_dist2(n, p) > best * 1.000001f) continue;       /* conservative: a few ulps of slack */
            if (n->b & 0x80000000u)
            {
                for (uint32_t k = 0; k < (n->b & 0x7FFFFFFFu); ++k)
                {
                    const uint32_t t = m->order[n->a + k];
                    const OClosest c = omesh_closest_simplex(p, omesh_vert(m, t, 0), omesh_vert(m, t, 1), omesh_vert(m, t, 2));
                    const mv3 d = mv_sub(p, c.pt);
                    const float d2 = mv_dot(d, d);
                    if (d2 < best || (d2 == best && t < bestTri)) { best = d2; bestTri = t; bestC = c; }
                }
            }
            else
            {
                const float dl = omesh_box_dist2(&m->nodes[n->a], p), dr = omesh_box_dist2(&m->nodes[n->b], p);
                if (dl <= dr) { if (sp < 63) stack[sp++] = n->b; stack[sp++] = n->a; }      /* nearer child on top */
                else          { if (sp < 63) stack[sp++] = n->a; stack[sp++] = n->b; }
            }
        }
    }
    if (bestTri == 0xFFFFFFFFu) return FLT_MAX;
    const mv3 pn = omesh_pseudo_normal(m, bestTri, bestC.simplex, bestC.id);
    const mv3 d = mv_sub(p, bestC.pt);
    const float sign = mv_dot(pn, d) > 0.0f ? 1.0f : -1.0f;               /* Mesh.cpp:61 */
    return sign * sqrtf(mv_dot(d, d));                                    /* Mesh.cpp:62 */
}

/* ---- construction ----------------------------------------------------------------------------------------- */
typedef struct { uint64_t key; uint32_t idx; } OEdge;
static int oedge_cmp(const void* a, const void* b)
{
    const OEdge* x = (const OEdge*)a; const OEdge* y = (const OEdge*)b;
    if (x->key != y->key) return x->key < y->key ? -1 : 1;
    return x->idx < y->idx ? -1 : (x->idx > y->idx);
}

static const float* g_omesh_cen; static int g_omesh_axis;
static int omesh_cen_cmp(const void* a, const void* b)
{
    const uint32_t x = *(const uint32_t*)a, y = *(const uint32_t*)b;
    const float cx = g_omesh_cen[3 * x + g_omesh_axis], cy = g_omesh_cen[3 * y + g_omesh_axis];
    if (cx != cy) return cx < cy ? -1 : 1;
    return x < y ? -1 : (x > y);
}

static uint32_t omesh_build_bvh(OMesh* m, const float* cen, const float* tmn, const float* tmx, uint32_t begin, uint32_t end)
{
    if (m->nNodes == m->capNodes) { m->capNodes = m->capNodes ? 2 * m->capNodes : 1024; m->nodes = (OBvhNode*)realloc(m->nodes, m->capNodes * sizeof(OBvhNode)); }
    const uint32_t idx = (uint32_t)m->nNodes++;
    float mn[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, mx[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX }, cmn[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, cmx[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
    for (uint32_t i = begin; i < end; ++i)
    {
        const uint32_t t = m->order[i];
        for (int d = 0; d < 3; ++d)
        {
            if (tmn[3 * t + d] < mn[d]) mn[d] = tmn[3 * t + d];
            if (tmx[3 * t + d] > mx[d]) mx[d] = tmx[3 * t + d];
            if (cen[3 * t + d] < cmn[d]) cmn[d] = cen[3 * t + d];
            if (cen[3 * t + d] > cmx[d]) cmx[d] = cen[3 * t + d];
        }
    }
    memcpy(m->nodes[idx].mn, mn, 12); memcpy(m->nodes[idx].mx, mx, 12);
    if (end - begin <= 4) { m->nodes[idx].a = begin; m->nodes[idx].b = 0x80000000u | (end - begin); return idx; }
    int axis = 0;
    if (cmx[1] - cmn[1] > cmx[axis] - cmn[axis]) axis = 1;
    if (cmx[2] - cmn[2] > cmx[axis] - cmn[axis]) axis = 2;
    g_omesh_cen = cen; g_omesh_axis = axis;
    qsort(m->order + begin, end - begin, sizeof(uint32_t), omesh_cen_cmp);
    const uint32_t mid = (begin + end) / 2;
    const uint32_t l = omesh_build_bvh(m, cen, tmn, tmx, begin, mid);
    const uint32_t r = omesh_build_bvh(m, cen, tmn, tmx, mid, end);
    m->nodes[idx].a = l; m->nodes[idx].b = r;
    return idx;
}

static void omesh_free(OMesh* m)
{
    if (!m) return;
    free(m->v); free(m->tri); free(m->he); free(m->nodes); free(m->order); free(m);
}

/* vertices: nv x 3 f32, tris: nt x 3 u32. Returns NULL if an edge has no twin (Mesh.cpp:121-128). */
static OMesh* omesh_create(const float* verts, size_t nv, const uint32_t* tris, size_t nt)
{
    OMesh* m = (OMesh*)calloc(1, sizeof(OMesh));
    m->nv = nv; m->nt = nt;
    m->v = (mv3*)malloc(nv * sizeof(mv3)); memcpy(m->v, verts, nv * 12);
    m->tri = (uint32_t*)malloc(3 * nt * 4); memcpy(m->tri, tris, 3 * nt * 4);
    m->he = (uint32_t*)malloc(3 * nt * 4); memset(m->he, 0xFF, 3 * nt * 4);
    /* CreateHalfEdges (Mesh.cpp:96-118) with a sort instead of the std::map: half-edges sorted by their UNDIRECTED edge, in
     * index order inside each run, then per run the map's find / insert sequence: "is the reverse edge stored? pair with it :
     * store this edge unless one of the same direction is already stored". On a non-manifold edge (more than two half-edges)
     * or a degenerate triangle (a, a, b) this can leave a half-edge unpaired, and the mesh is rejected as the reference does. */
    OEdge* e = (OEdge*)malloc(3 * nt * sizeof(OEdge));
    for (uint32_t i = 0; i < 3 * nt; ++i)
    {
        const uint32_t a = m->tri[i], b = (i % 3 == 2) ? m->tri[i - 2] : m->tri[i + 1];
        e[i].key = a < b ? (((uint64_t)a << 32) | b) : (((uint64_t)b << 32) | a); e[i].idx = i;
    }
    qsort(e, 3 * nt, sizeof(OEdge), oedge_cmp);
    for (size_t r = 0; r < 3 * nt;)
    {
        const uint32_t lo = (uint32_t)(e[r].key >> 32);
        uint32_t stored[2] = { 0xFFFFFFFFu, 0xFFFFFFFFu };                 /* [0] lo -> hi, [1] hi -> lo */
        size_t q = r;
        for (; q < 3 * nt && e[q].key == e[r].key; ++q)
        {
            const uint32_t i = e[q].idx, dir = m->tri[i] == lo ? 0u : 1u;
            if (stored[dir ^ 1u] != 0xFFFFFFFFu) { m->he[stored[dir ^ 1u]] = i; m->he[i] = stored[dir ^ 1u]; }
            else if (stored[dir] == 0xFFFFFFFFu) stored[dir] = i;
        }
        r = q;
    }
    free(e);
    for (uint32_t i = 0; i < 3 * nt; ++i) if (m->he[i] == 0xFFFFFFFFu) { omesh_free(m); return NULL; }
    float* cen = (float*)malloc(3 * nt * 4); float* tmn = (float*)malloc(3 * nt * 4); float* tmx = (float*)malloc(3 * nt * 4);
    m->order = (uint32_t*)malloc(nt * 4);
    for (uint32_t t = 0; t < nt; ++t)
    {
        m->order[t] = t;
        for (int d = 0; d < 3; ++d)
        {
            float lo = FLT_MAX, hi = -FLT_MAX;
            for (int k = 0; k < 3; ++k) { const mv3 p = omesh_vert(m, t, (uint32_t)k); const float c = d == 0 ? p.x : d == 1 ? p.y : p.z; if (c < lo) lo = c; if (c > hi) hi = c; }
            tmn[3 * t + d] = lo; tmx[3 * t + d] = hi; cen[3 * t + d] = 0.5f * (lo + hi);
        }
    }
    omesh_build_bvh(m, cen, tmn, tmx, 0, (uint32_t)nt);
    free(cen); free(tmn); free(tmx);
    return m;
}

#endif
