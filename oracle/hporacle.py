"""ctypes bindings of oracle/_build/libhporacle.so — the plain-C restatement (oracle/hp_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg.
The product (hp-adaptive-signed-distance-field-octree_b200/) never imports this.
"""
import ctypes as C
import os
import subprocess
import numpy as np

from .hpref import Config, Instr, make_config, make_program, parse_block, canonical, STAT_KEYS, NCOEF  # noqa: F401

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "_build", "libhporacle.so")


def build():
    """Compile the restatement (gcc, seconds). Building the checker is not using it."""
    subprocess.check_call(["make", "-C", HERE, "port"], stdout=subprocess.DEVNULL)


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO):
        build()
    L = C.CDLL(SO)
    L.hporacle_build.restype = C.c_void_p
    L.hporacle_build.argtypes = [C.POINTER(Config), C.POINTER(Instr), C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                 C.c_double, C.c_int, C.c_void_p]
    L.hporacle_destroy.argtypes = [C.c_void_p]
    L.hporacle_block_size.restype = C.c_size_t
    L.hporacle_block_size.argtypes = [C.c_void_p]
    L.hporacle_block_copy.argtypes = [C.c_void_p, C.c_void_p]
    L.hporacle_from_block.restype = C.c_void_p
    L.hporacle_from_block.argtypes = [C.c_void_p, C.c_size_t]
    L.hporacle_query.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int]
    L.hporacle_query_gradient.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_int]
    L.hporacle_query_ray.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_double, C.c_void_p, C.c_void_p]
    L.hporacle_stats.argtypes = [C.c_void_p, C.c_void_p]
    L.hporacle_apply_log.argtypes = [C.c_void_p, C.c_void_p]
    L.hporacle_fit.restype = C.c_double
    L.hporacle_fit.argtypes = [C.POINTER(Config), C.POINTER(Instr), C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32,
                               C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]
    L.hporacle_sdf_eval_batch.argtypes = [C.POINTER(Instr), C.c_uint32, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
    L.hporacle_continuity_csr.restype = C.c_size_t
    L.hporacle_continuity_csr.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    L.hporacle_n_coeffs.restype = C.c_size_t
    L.hporacle_n_coeffs.argtypes = [C.c_void_p]
    L.hporacle_n_nodes.restype = C.c_size_t
    L.hporacle_n_nodes.argtypes = [C.c_void_p]
    L.hporacle_tables.argtypes = [C.c_void_p] * 7
    L.hporacle_mesh_create.restype = C.c_void_p
    L.hporacle_mesh_create.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
    L.hporacle_mesh_destroy.argtypes = [C.c_void_p]
    L.hporacle_mesh_sdf.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int]
    L.hporacle_mesh_half_edges.argtypes = [C.c_void_p, C.c_void_p]
    L.hporacle_set_nearness_mc.argtypes = [C.c_int, C.c_uint64]
    _lib = L
    return L


class OracleTree:
    """Deterministic strict-greedy build (exact-mean nearness) by the C restatement."""

    def __init__(self, handle, keep=()):
        self.h, self._keep = handle, keep

    @classmethod
    def build(cls, cfg, prog, max_degree=11, max_depth=10, total_mode=0, cg_tol=0.0, threads=1, mc_seed=None):
        """mc_seed: None = exact-mean nearness; an integer = the 100-sample estimator on Philox points (mc_counter)."""
        lib().hporacle_set_nearness_mc(0 if mc_seed is None else 1, 0 if mc_seed is None else mc_seed)
        try:
            h = lib().hporacle_build(C.byref(cfg), prog, len(prog), max_degree, max_depth, total_mode, cg_tol, threads, None)
        finally:
            lib().hporacle_set_nearness_mc(0, 0)
        return cls(h, keep=(prog,))

    @classmethod
    def from_block(cls, block):
        buf = np.frombuffer(bytes(block), dtype=np.uint8).copy()
        h = lib().hporacle_from_block(buf.ctypes.data, buf.size)
        if not h:
            raise ValueError("MemoryBlock does not parse")
        return cls(h)

    def block(self):
        n = lib().hporacle_block_size(self.h)
        buf = np.empty(n, dtype=np.uint8)
        lib().hporacle_block_copy(self.h, buf.ctypes.data)
        return buf

    def query(self, pts, threads=1):
        pts = np.ascontiguousarray(pts, dtype=np.float64)
        out = np.empty(len(pts), dtype=np.float64)
        lib().hporacle_query(self.h, pts.ctypes.data, len(pts), out.ctypes.data, threads)
        return out

    def query_gradient(self, pts, threads=1):
        pts = np.ascontiguousarray(pts, dtype=np.float64)
        out = np.empty(len(pts), dtype=np.float64)
        g = np.empty((len(pts), 3), dtype=np.float64)
        lib().hporacle_query_gradient(self.h, pts.ctypes.data, len(pts), out.ctypes.data, g.ctypes.data, threads)
        return out, g

    def query_ray(self, origins, dirs, t_max):
        o = np.ascontiguousarray(origins, np.float64)
        d = np.ascontiguousarray(dirs, np.float64)
        hit = np.zeros(len(o), np.uint8)
        t = np.zeros(len(o), np.float64)
        lib().hporacle_query_ray(self.h, o.ctypes.data, d.ctypes.data, len(o), float(t_max), hit.ctypes.data, t.ctypes.data)
        return hit.astype(bool), t

    def stats(self):
        s = np.zeros(10)
        lib().hporacle_stats(self.h, s.ctypes.data)
        return dict(zip(STAT_KEYS, s.tolist()))

    def apply_log(self):
        n = int(self.stats()["log_size"])
        a = np.zeros((n, 8))
        if n:
            lib().hporacle_apply_log(self.h, a.ctypes.data)
        return a

    def continuity_csr(self, with_diagonal=False):
        L = lib()
        n = L.hporacle_n_coeffs(self.h)
        nnz = L.hporacle_continuity_csr(self.h, int(with_diagonal), None, None, None)
        rp = np.empty(n + 1, np.int64)
        col = np.empty(nnz, np.int32)
        val = np.empty(nnz, np.float64)
        L.hporacle_continuity_csr(self.h, int(with_diagonal), rp.ctypes.data, col.ctypes.data, val.ctypes.data)
        return rp, col, val

    def close(self):
        if self.h:
            lib().hporacle_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class OracleMesh:
    """Float32 mesh signed distance (Mesh::SignedDistanceAtPt restated); `h` can be the handle of a ("mesh", [], h) item."""

    def __init__(self, verts, tris):
        self.v = np.ascontiguousarray(verts, np.float32)
        self.t = np.ascontiguousarray(tris, np.uint32)
        self.h = lib().hporacle_mesh_create(self.v.ctypes.data, len(self.v), self.t.ctypes.data, len(self.t))
        if not self.h:
            raise ValueError("mesh is not a closed manifold")

    def sdf(self, pts, use_bvh=True, threads=1):
        p = np.ascontiguousarray(pts, np.float32)
        out = np.empty(len(p), np.float32)
        lib().hporacle_mesh_sdf(self.h, p.ctypes.data, len(p), out.ctypes.data, 1 if use_bvh else 0, threads)
        return out

    def half_edges(self):
        """Twin of every half-edge (3 per triangle, half-edge 3t + k runs from vertex k to vertex k + 1 of triangle t)."""
        out = np.empty(3 * len(self.t), np.uint32)
        lib().hporacle_mesh_half_edges(self.h, out.ctypes.data)
        return out

    def close(self):
        if self.h:
            lib().hporacle_mesh_destroy(self.h)
            self.h = None


def oracle_fit(cfg, prog, aabb_min, aabb_max, degree, depth, degree_in=0, coeffs_in=None):
    """FitPolynomial restatement, nearness None -> (coeffs[N_degree], raw_err)."""
    out = np.zeros(NCOUNT[degree])
    mn = np.asarray(aabb_min, np.float32)
    mx = np.asarray(aabb_max, np.float32)
    cin = np.ascontiguousarray(coeffs_in, np.float64) if coeffs_in is not None else np.zeros(1)
    err = lib().hporacle_fit(C.byref(cfg), prog, len(prog), mn.ctypes.data, mx.ctypes.data, degree_in, cin.ctypes.data,
                             degree, depth, out.ctypes.data, None)
    return out, err


def sdf_eval(prog, pts):
    pts = np.ascontiguousarray(pts, np.float64)
    out = np.empty(len(pts))
    lib().hporacle_sdf_eval_batch(prog, len(prog), pts.ctypes.data, len(pts), out.ctypes.data, None)
    return out


def tables():
    t = dict(nl=np.zeros((13, 11)), counts=np.zeros(13, np.uint32), basis_idx=np.zeros((455, 3), np.uint32),
             recur=np.zeros((13, 2)), roots=np.zeros(2080), weights=np.zeros(2080), face_lookup=np.zeros((3, 4, 2), np.uint32))
    lib().hporacle_tables(*[t[k].ctypes.data for k in ("nl", "counts", "basis_idx", "recur", "roots", "weights", "face_lookup")])
    return t


# LegendreCoeffientCount with the reference's truncation quirk at degree 6 (Utility.h:87-106 gives 83, not 84)
NCOUNT = [1, 4, 10, 20, 35, 56, 83, 120, 165, 220, 286, 364, 455]
