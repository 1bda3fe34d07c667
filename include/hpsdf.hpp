// hpsdf.hpp — C++ host facade with the reference's public surface, forwarding to the C ABI (hpsdf.h).
//
// Mirrors (names, argument meaning, ownership) of jw007123/hp-Adaptive-Signed-Distance-Field-Octree:
//     SDF::Config                 Include/HP/Config.h:12-43        (same members, same 80-byte LP64 image)
//     SDF::Octree                 Include/HP/Octree.h:36-86        Create / Query / QueryWithGradient / QueryRay / UnionSDF /
//                                                                  SubtractSDF / IntersectSDF / Clear / FromMemoryBlock /
//                                                                  ToMemoryBlock / GetRootAABB, copy + move; plus
//                                                                  ExtractIsosurface / Raycast / RaycastDevice /
//                                                                  QueryDerivatives / QueryDerivativesDevice (no
//                                                                  counterpart in the reference)
//     MemoryBlock                 Include/Utility/MemoryBlock.h:5-9
//
// Differences, all forced by the device: (1) Create takes an SDF::Program (closed-form primitives / meshes / trees
// combined by union, intersection, difference — evaluated on the GPU) where the reference takes a
// std::function<f64(const Eigen::Vector3d&, u32)>; arbitrary host lambdas stay on the reference's CPU path and the
// std::function overload here throws. (2) Query has a batch overload (the reference's callers loop). (3) Errors are
// exceptions (SDF::Error with the hpsdf_status) where the reference asserts.
//
// Vector / box arguments are templates over anything with x()/y()/z() (points) or min()/max() (boxes), so call sites
// written against Eigen compile unchanged; Eigen itself is not required. Header-only; link with libhpsdf.so.
#pragma once
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>
#include <stdexcept>
#include <string>
#include <thread>
#include <utility>
#include <vector>
#include "hpsdf.h"

// The reference's literal types (Include/Utility/Literals.h): u32 is `long unsigned int` there, 8 bytes on LP64.
struct MemoryBlock
{
    size_t size;
    void*  ptr;
};

namespace SDF
{
    struct Error : std::runtime_error
    {
        hpsdf_status status;
        Error(hpsdf_status s, const std::string& what) : std::runtime_error(what), status(s) {}
    };

    inline void check(hpsdf_status s)
    {
        if (s != HPSDF_OK) throw Error(s, std::string(hpsdf_status_string(s)) + ": " + hpsdf_last_error());
    }

    // Minimal 3-vector / box used where the reference uses Eigen::Vector3d / Eigen::AlignedBox3f.
    struct Vec3d { double v[3]; double x() const { return v[0]; } double y() const { return v[1]; } double z() const { return v[2]; } };
    struct Box3f
    {
        float lo[3], hi[3];
        struct Corner { float* p; float& operator()(int i) { return p[i]; } float x() const { return p[0]; } float y() const { return p[1]; } float z() const { return p[2]; } };
        Corner min() { return Corner{ lo }; }
        Corner max() { return Corner{ hi }; }
    };

    // SDF::Config with the reference's member names; bit-compatible with hpsdf_config / the MemoryBlock tail.
    struct Config
    {
        struct NearnessWeighting
        {
            enum Type : uint8_t { None = 0, Polynomial = 1, Exponential = 2 } type;
            double strength;
        } nearnessWeighting;

        struct Continuity
        {
            bool   enforce;
            double strength;
        } continuity;

        bool          enableLogging;
        double        targetErrorThreshold;
        unsigned long threadCount;
        Box3f         root;

        Config()                                                     // Config::Config (Config.cpp:5-14)
        {
            hpsdf_config c;
            hpsdf_config_default(&c);
            std::memcpy(static_cast<void*>(this), &c, sizeof(c));
        }
        void IsValid() const { check(hpsdf_config_validate(reinterpret_cast<const hpsdf_config*>(this))); }   // Config.cpp:17-32
        template <class Box> void SetRoot(const Box& b)
        {
            root.lo[0] = b.min().x(); root.lo[1] = b.min().y(); root.lo[2] = b.min().z();
            root.hi[0] = b.max().x(); root.hi[1] = b.max().y(); root.hi[2] = b.max().z();
        }
        const hpsdf_config* c() const { return reinterpret_cast<const hpsdf_config*>(this); }
    };
    static_assert(sizeof(Config) == sizeof(hpsdf_config) && sizeof(Config) == 80, "SDF::Config must keep the reference's 80-byte layout");

    class Octree;

    /// R(t) = O + t * D with |D| = 1 (Include/HP/Ray.h:10-24)
    struct Ray { Vec3d origin, direction; };

    // Device SDF: postfix program of primitives and boolean operators (see hpsdf.h).
    class Program
    {
    public:
        Program& Sphere(double cx, double cy, double cz, double r) { return push(HPSDF_PRIM_SPHERE, { cx, cy, cz, r }); }
        Program& Box(double cx, double cy, double cz, double hx, double hy, double hz) { return push(HPSDF_PRIM_BOX, { cx, cy, cz, hx, hy, hz }); }
        Program& Torus(double cx, double cy, double cz, double R, double r, int axis) { return push(HPSDF_PRIM_TORUS, { cx, cy, cz, R, r, (double)axis }); }
        Program& Capsule(double ax, double ay, double az, double bx, double by, double bz, double r) { return push(HPSDF_PRIM_CAPSULE, { ax, ay, az, bx, by, bz, r }); }
        Program& Plane(double nx, double ny, double nz, double d) { return push(HPSDF_PRIM_PLANE, { nx, ny, nz, d }); }
        Program& Mesh(const hpsdf_mesh* m) { return push(HPSDF_PRIM_MESH, {}, m); }
        inline Program& Tree(const Octree& t);
        Program& Union() { return push(HPSDF_OP_UNION, {}); }             // min(a, b)
        Program& Intersect() { return push(HPSDF_OP_INTERSECT, {}); }     // max(a, b)
        Program& Subtract() { return push(HPSDF_OP_SUBTRACT, {}); }       // max(a, -b)
        Program& Negate() { return push(HPSDF_OP_NEGATE, {}); }
        Program& Append(const Program& o) { instr_.insert(instr_.end(), o.instr_.begin(), o.instr_.end()); return *this; }
        hpsdf_sdf_program c() const { return hpsdf_sdf_program{ (uint32_t)instr_.size(), 0u, instr_.data() }; }

    private:
        std::vector<hpsdf_sdf_instr> instr_;
        Program& push(uint32_t op, std::initializer_list<double> p, const void* handle = nullptr)
        {
            hpsdf_sdf_instr in;
            std::memset(&in, 0, sizeof(in));
            in.op = op; in.handle = handle;
            int k = 0;
            for (double v : p) in.p[k++] = v;
            instr_.push_back(in);
            return *this;
        }
    };

    class Octree
    {
    public:
        Octree() = default;
        ~Octree() { Clear(); }
        Octree(const Octree& o) { if (o.h_) check(hpsdf_clone(o.h_, &h_)); }                           // Octree.cpp:24-45
        Octree(Octree&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }                                     // Octree.cpp:76-86
        Octree& operator=(const Octree& o) { if (this != &o) { Clear(); if (o.h_) check(hpsdf_clone(o.h_, &h_)); } return *this; }
        Octree& operator=(Octree&& o) noexcept { if (this != &o) { Clear(); h_ = o.h_; o.h_ = nullptr; } return *this; }

        /// Approximates F_ using the parameters in config_ (Octree.cpp:312-352). Blocks; runs on the GPU.
        void Create(const Config& config_, const Program& F_, const hpsdf_build_opts* opts_ = nullptr)
        {
            Clear();
            const hpsdf_sdf_program p = F_.c();
            check(hpsdf_create(config_.c(), opts_, &p, &h_));
        }
        /// The reference's signature. Host callables cannot run on the device: they remain the reference's CPU path.
        void Create(const Config&, std::function<double(const Vec3d&, const unsigned long)>)
        {
            throw Error(HPSDF_ERR_UNSUPPORTED, "Create(std::function): arbitrary host lambdas stay on the reference's CPU path; pass an SDF::Program");
        }

        /// Resultant SDF = Min(oldF, F_) / Max(F_, -oldF) / Max(oldF, F_)   (Octree.cpp:355-400)
        /// opts_ (optional) carries what the reference fixes at compile time (max degree / depth, ...); the rebuild runs on the
        /// old tree's device unless opts_->device names one. If the rebuild fails the tree is left as it was.
        void UnionSDF(const Program& F_, const hpsdf_build_opts* opts_ = nullptr)     { combine(F_, HPSDF_OP_UNION, opts_); }
        void SubtractSDF(const Program& F_, const hpsdf_build_opts* opts_ = nullptr)  { combine(F_, HPSDF_OP_SUBTRACT, opts_); }
        void IntersectSDF(const Program& F_, const hpsdf_build_opts* opts_ = nullptr) { combine(F_, HPSDF_OP_INTERSECT, opts_); }

        /// Resets the tree (Octree.cpp:459-471)
        void Clear() { if (h_) hpsdf_destroy(h_); h_ = nullptr; }

        /// Creates an octree from a previously serialised version; the caller keeps the block (Octree.cpp:403-421)
        void FromMemoryBlock(MemoryBlock octBlock_, int device_ = -1)
        {
            Clear();
            check(hpsdf_from_memory_block(octBlock_.ptr, octBlock_.size, device_, &h_));
        }
        /// Serialises an octree to a memory block owned by malloc: the caller free()s ptr (Octree.cpp:424-456)
        MemoryBlock ToMemoryBlock() const
        {
            MemoryBlock b = { 0, nullptr };
            check(hpsdf_to_memory_block(need(), &b.size, &b.ptr));
            return b;
        }

        /// Distance from F = 0, negative inside; DBL_MAX outside the root (Octree.cpp:662-702)
        template <class V3> double Query(const V3& pt_) const
        {
            const double xyz[3] = { pt_.x(), pt_.y(), pt_.z() };
            double out = 0.0;
            check(hpsdf_query(need(), xyz, 1, &out));
            return out;
        }
        /// Batched form: xyz_ = n x 3 doubles (what an array of Eigen::Vector3d is), out_ = n doubles; host pointers.
        void Query(const double* xyz_, size_t n_, double* out_) const { check(hpsdf_query(need(), xyz_, n_, out_)); }
        /// Device pointers, asynchronous on a cudaStream_t.
        void QueryDevice(const double* dXyz_, size_t n_, double* dOut_, void* stream_) const { check(hpsdf_query_device(need(), dXyz_, n_, dOut_, stream_)); }

        /// As Query, with the unit gradient by central differences (Octree.cpp:749-789)
        template <class V3> double QueryWithGradient(const V3& pt_, V3& unitNormal_) const
        {
            const double xyz[3] = { pt_.x(), pt_.y(), pt_.z() };
            double out = 0.0, g[3] = { 0, 0, 0 };
            check(hpsdf_query_with_gradient(need(), xyz, 1, &out, g));
            unitNormal_ = V3{ g[0], g[1], g[2] };
            return out;
        }

        /// Sphere-traces the field along a ray (Octree.cpp:705-746); `Ray` is anything with .origin and .direction (x()/y()/z()),
        /// e.g. SDF::Ray below or the reference's own struct
        template <class RayT> bool QueryRay(const RayT& ray_, const double tMax_, double& t_) const
        {
            const double o[3] = { ray_.origin.x(), ray_.origin.y(), ray_.origin.z() };
            const double d[3] = { ray_.direction.x(), ray_.direction.y(), ray_.direction.z() };
            unsigned char hit = 0;
            double t = 0.0;
            check(hpsdf_query_ray(need(), o, d, 1, tMax_, &hit, &t));
            if (hit) t_ = t;                                             // the reference writes t_ only when it returns true (:733)
            return hit != 0;
        }
        void QueryRay(const double* origins_, const double* directions_, size_t n_, double tMax_, unsigned char* hit_, double* t_) const
        {
            check(hpsdf_query_ray(need(), origins_, directions_, n_, tMax_, hit_, t_));
        }

        /// First crossing of F = iso_ along n_ rays o + t d, t in [tMin_, tMax_] (hpsdf_raycast): tHit_ gets t or +INFINITY for a
        /// miss, normals_ (3 per ray, may be nullptr) the unit gradient of the hit leaf's polynomial. The ray query to use.
        void Raycast(const double* origins_, const double* directions_, size_t n_, double tMin_, double tMax_, double iso_, double* tHit_,
                     double* normals_ = nullptr) const
        {
            check(hpsdf_raycast(need(), origins_, directions_, n_, tMin_, tMax_, iso_, tHit_, normals_));
        }

        /// Raycast with device pointers, asynchronous on stream_ (hpsdf_raycast_device).
        void RaycastDevice(const double* dOrigins_, const double* dDirections_, size_t n_, double tMin_, double tMax_, double iso_,
                           double* dTHit_, double* dNormals_, void* stream_) const
        {
            check(hpsdf_raycast_device(need(), dOrigins_, dDirections_, n_, tMin_, tMax_, iso_, dTHit_, dNormals_, stream_));
        }

        /// Query's value with the exact gradient and, when hess_ is not nullptr, Hessian (xx, xy, xz, yy, yz, zz) of the hit leaf's
        /// polynomial in user space, not normalised; 0 outside the root (hpsdf_query_derivatives). Host pointers, n_ x 3 points.
        void QueryDerivatives(const double* xyz_, size_t n_, double* value_, double* grad_, double* hess_ = nullptr) const
        {
            check(hpsdf_query_derivatives(need(), xyz_, n_, value_, grad_, hess_));
        }

        /// QueryDerivatives with device pointers, asynchronous on stream_ (hpsdf_query_derivatives_device).
        void QueryDerivativesDevice(const double* dXyz_, size_t n_, double* dValue_, double* dGrad_, double* dHess_, void* stream_) const
        {
            check(hpsdf_query_derivatives_device(need(), dXyz_, n_, dValue_, dGrad_, dHess_, stream_));
        }

        /// The level set F = iso_ as a triangle mesh (hpsdf_extract_isosurface): marching tetrahedra over resolution_ cells per axis
        /// spanning [boxMin_, boxMax_] (both nullptr = the root box). vertices_ gets 3 floats per vertex, triIndices_ 3 indices per
        /// triangle, counter-clockwise seen from the side where F >= iso_: what Meshing::Mesh::Create takes.
        void ExtractIsosurface(const uint32_t resolution_[3], double iso_, std::vector<float>& vertices_, std::vector<uint32_t>& triIndices_,
                               const double* boxMin_ = nullptr, const double* boxMax_ = nullptr) const
        {
            size_t nv = 0, nt = 0;
            float* v = nullptr;
            uint32_t* t = nullptr;
            check(hpsdf_extract_isosurface(need(), resolution_, boxMin_, boxMax_, iso_, &nv, &v, &nt, &t));
            std::unique_ptr<float, void (*)(void*)> ownV(v, std::free);
            std::unique_ptr<uint32_t, void (*)(void*)> ownT(t, std::free);
            vertices_.assign(v, v + 3 * nv);
            triIndices_.assign(t, t + 3 * nt);
        }

        /// The aabb of the root node (Octree.cpp:106-109)
        Box3f GetRootAABB() const { Box3f b; check(hpsdf_get_root_aabb(need(), b.lo, b.hi)); return b; }

        hpsdf_build_stats Stats() const { hpsdf_build_stats s; check(hpsdf_get_build_stats(need(), &s)); return s; }
        const hpsdf_octree* handle() const { return h_; }

    private:
        hpsdf_octree* h_ = nullptr;
        const hpsdf_octree* need() const { if (!h_) throw Error(HPSDF_ERR_INVALID_ARG, "octree is empty"); return h_; }
        void combine(const Program& F_, uint32_t op_, const hpsdf_build_opts* opts_)
        {
            Octree oldTree = std::move(*this);                          // keeps the old tree alive until Create returns (Octree.cpp:366)
            try
            {
                Config cfg;
                check(hpsdf_get_config(oldTree.need(), reinterpret_cast<hpsdf_config*>(&cfg)));
                hpsdf_build_opts o;
                if (opts_) o = *opts_; else hpsdf_build_opts_default(&o);
                if (o.device < 0) check(hpsdf_get_device(oldTree.need(), &o.device));
                Program p;
                p.Append(F_).Tree(oldTree);
                if (op_ == HPSDF_OP_UNION) p.Union(); else if (op_ == HPSDF_OP_INTERSECT) p.Intersect(); else p.Subtract();
                Create(cfg, p, &o);
            }
            catch (...)
            {
                *this = std::move(oldTree);                             // a failed rebuild leaves the tree as it was
                throw;
            }
        }
    };

    inline Program& Program::Tree(const Octree& t) { return push(HPSDF_PRIM_OCTREE, {}, t.handle()); }
}

// Meshing::Mesh (Include/Meshing/Mesh.h:43-99) + Meshing::BVH as an SDF source on the device. The OBJ reader stays the
// reference's: hand over its `vertices` / `triIndices` arrays. Create() does what CreateFromObj does after parsing
// (CreateHalfEdges, Mesh.cpp:87-131; false for a mesh that is not a closed manifold) and what BVH::Create does, on the host,
// then uploads; SignedDistanceAtPt is the BVH overload of Mesh.cpp:54-63 (float32, bit-identical).
namespace Meshing
{
    class Mesh
    {
    public:
        Mesh() = default;
        Mesh(const Mesh&) = delete;
        Mesh& operator=(const Mesh&) = delete;
        ~Mesh() { Clear(); }
        void Clear() { if (h_) hpsdf_mesh_destroy(h_); h_ = nullptr; }

        /// xyz_: 3 floats per vertex; triIndices_: 3 indices per triangle, counter-clockwise seen from outside
        bool Create(const float* xyz_, size_t nVertices_, const uint32_t* triIndices_, size_t nTriangles_, int device_ = -1)
        {
            Clear();
            const hpsdf_status st = hpsdf_mesh_create(xyz_, nVertices_, triIndices_, nTriangles_, device_, &h_);
            if (st == HPSDF_ERR_MESH) return false;                         // the reference's CreateHalfEdges returns false
            if (st != HPSDF_OK) throw SDF::Error(st, hpsdf_last_error());
            return true;
        }
        /// > 0 implies outside mesh
        float SignedDistanceAtPt(float x_, float y_, float z_) const
        {
            const float p[3] = { x_, y_, z_ };
            float d = 0.0f;
            const hpsdf_status st = hpsdf_mesh_signed_distance(need(), p, 1, &d);
            if (st != HPSDF_OK) throw SDF::Error(st, hpsdf_last_error());
            return d;
        }
        void SignedDistanceAtPts(const float* xyz_, size_t n_, float* out_) const
        {
            const hpsdf_status st = hpsdf_mesh_signed_distance(need(), xyz_, n_, out_);
            if (st != HPSDF_OK) throw SDF::Error(st, hpsdf_last_error());
        }
        SDF::Box3f CalculateMeshAABB() const
        {
            SDF::Box3f b;
            const hpsdf_status st = hpsdf_mesh_aabb(need(), b.lo, b.hi);
            if (st != HPSDF_OK) throw SDF::Error(st, hpsdf_last_error());
            return b;
        }
        const hpsdf_mesh* handle() const { return h_; }

    private:
        hpsdf_mesh* h_ = nullptr;
        const hpsdf_mesh* need() const { if (!h_) throw SDF::Error(HPSDF_ERR_INVALID_ARG, "mesh is empty"); return h_; }
    };
}
