"""hpsdf_b200 — host-side mirror of the reference's public surface over the C ABI (include/hpsdf.h).

Names, argument meaning and error behaviour follow the reference (SDF::Config, SDF::Octree::Create / Query /
ToMemoryBlock / FromMemoryBlock / Clear / GetRootAABB, MemoryBlock; Include/HP/Octree.h:36-86, Include/HP/Config.h,
Include/Utility/MemoryBlock.h) so parity tests read like the reference's own (Source/Tests/HPUnitTests.cpp).
The one difference is what replaces the std::function argument of Create: a device SDF program (`SdfProgram`).

Everything here is ctypes over `lib/libhpsdf.so` (CUDA, sm_100a). There is NO CPU fallback: if the library is missing
or no GPU is present the calls raise. This module never imports anything under oracle/.

Load it with importlib (the directory name has hyphens):
    hp = importlib.import_module("hp-adaptive-signed-distance-field-octree_b200")
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HPSDF_LIB", os.path.join(HERE, "lib", "libhpsdf.so"))

# ---- enums (include/hpsdf.h) ---------------------------------------------------------------------------------------
OK, ERR_INVALID_ARG, ERR_NO_DEVICE, ERR_CUDA, ERR_BAD_BLOCK, ERR_UNSUPPORTED, ERR_COMM, ERR_OOM, ERR_MESH = range(9)
NEARNESS_NONE, NEARNESS_POLYNOMIAL, NEARNESS_EXPONENTIAL = 0, 1, 2
TOTAL_REFERENCE, TOTAL_EXACT_SUM = 0, 1
NEARNESS_EXACT_MEAN, NEARNESS_MC_COUNTER = 0, 1      # hpsdf_build_opts.nearness_mode
CG_GUESS_COEFFS, CG_GUESS_REFERENCE = 0, 1           # hpsdf_build_opts.cg_guess
PRIM = dict(sphere=1, box=2, torus=3, capsule=4, plane=5, mesh=16, octree=17)
OP = dict(union=64, intersect=65, subtract=66, negate=67)
# LegendreCoeffientCount incl. the reference's f64 truncation at degree 6 (Utility.h:87-106 yields 83, not 84)
COEFF_COUNT = [1, 4, 10, 20, 35, 56, 83, 120, 165, 220, 286, 364, 455]
INTERNAL_TAG = 13
DBL_MAX = np.finfo(np.float64).max


class HpsdfError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("hpsdf status %d: %s" % (status, message))
        self.status = status


class Config(C.Structure):
    """SDF::Config, 80-byte LP64 image (Include/HP/Config.h:12-43). Field names follow the reference's members."""
    _fields_ = [("nearness_type", C.c_uint8), ("_pad0", C.c_uint8 * 7), ("nearness_strength", C.c_double),
                ("continuity_enforce", C.c_uint8), ("_pad1", C.c_uint8 * 7), ("continuity_strength", C.c_double),
                ("enable_logging", C.c_uint8), ("_pad2", C.c_uint8 * 7), ("target_error_threshold", C.c_double),
                ("thread_count", C.c_uint64), ("root_min", C.c_float * 3), ("root_max", C.c_float * 3)]

    def __init__(self, **kw):
        super().__init__()
        lib().hpsdf_config_default(C.byref(self))          # Config::Config() (Config.cpp:5-14)
        for k, v in kw.items():
            if k in ("root_min", "root_max"):
                getattr(self, k)[:] = [float(np.float32(x)) for x in v]
            else:
                setattr(self, k, v)

    def IsValid(self):
        """Config::IsValid (Config.cpp:17-32): raises instead of asserting."""
        _check(lib().hpsdf_config_validate(C.byref(self)))


class BuildOpts(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("max_degree", C.c_uint32), ("max_depth", C.c_uint32),
                ("nearness_mode", C.c_uint32), ("total_mode", C.c_uint32), ("cg_max_iterations", C.c_uint32),
                ("cg_tolerance", C.c_double), ("device", C.c_int32), ("speculate", C.c_uint32),
                ("strict_order", C.c_uint32), ("comm", C.c_void_p), ("stream", C.c_void_p),
                ("jit", C.c_uint32), ("min_round_jobs", C.c_uint32), ("scheduler", C.c_uint32), ("cg_guess", C.c_uint32),
                ("nearness_seed", C.c_uint64)]

    def __init__(self, **kw):
        super().__init__()
        lib().hpsdf_build_opts_default(C.byref(self))
        for k, v in kw.items():
            setattr(self, k, v)


class Instr(C.Structure):
    _fields_ = [("op", C.c_uint32), ("_pad", C.c_uint32), ("handle", C.c_void_p), ("p", C.c_double * 8)]


class _Program(C.Structure):
    _fields_ = [("n_instr", C.c_uint32), ("_pad", C.c_uint32), ("instr", C.POINTER(Instr))]


class BuildStats(C.Structure):
    _fields_ = [("n_nodes", C.c_uint64), ("n_leaves", C.c_uint64), ("n_coeffs", C.c_uint64), ("rounds", C.c_uint64),
                ("jobs_evaluated", C.c_uint64), ("jobs_applied_p", C.c_uint64), ("jobs_applied_h", C.c_uint64),
                ("fits_evaluated", C.c_uint64), ("sdf_evals", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("algorithmic_flops", C.c_double), ("sdf_flops_per_eval", C.c_double), ("total_error", C.c_double), ("exact_total_error", C.c_double),
                ("cut_margin", C.c_double), ("fit_kernel_ms", C.c_double), ("continuity_ms", C.c_double), ("continuity_enum_ms", C.c_double),
                ("continuity_assembly_ms", C.c_double), ("continuity_cg_ms", C.c_double),
                ("host_replay_ms", C.c_double), ("host_select_ms", C.c_double), ("host_tasks_ms", C.c_double),
                ("device_wait_ms", C.c_double), ("pack_ms", C.c_double), ("finalize_ms", C.c_double), ("total_ms", C.c_double), ("cg_iterations", C.c_uint64),
                ("cg_relative_residual", C.c_double), ("near_tie_decisions", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class DecisionLogEntry(C.Structure):
    _fields_ = [("node_idx", C.c_uint64), ("depth", C.c_uint32), ("degree", C.c_uint32), ("centre", C.c_float * 3),
                ("chose_p", C.c_uint32), ("kind", C.c_uint32), ("p_improvement", C.c_double),
                ("h_improvement", C.c_double), ("relative_margin", C.c_double)]


class ApplyLogEntry(C.Structure):
    _fields_ = [("node_idx", C.c_uint64), ("kind", C.c_uint32), ("degree", C.c_uint32), ("initial_err", C.c_double),
                ("new_err", C.c_double), ("p_improvement", C.c_double), ("h_improvement", C.c_double),
                ("total_after", C.c_double)]


class FrontierBench(C.Structure):
    _fields_ = [("ms_per_launch", C.c_double), ("jobs", C.c_uint64), ("fits", C.c_uint64), ("sdf_evals", C.c_uint64),
                ("algorithmic_flops", C.c_double), ("sdf_flops_per_eval", C.c_double), ("checksum", C.c_double)]


assert C.sizeof(Config) == 80 and C.sizeof(Instr) == 80

# every symbol include/hpsdf.h declares (tests/test_abi.py checks the library exports them all)
EXPORTS = [
    "hpsdf_status_string", "hpsdf_last_error", "hpsdf_version", "hpsdf_device_count", "hpsdf_config_default",
    "hpsdf_config_validate", "hpsdf_build_opts_default", "hpsdf_sdf_eval", "hpsdf_mesh_create",
    "hpsdf_mesh_signed_distance", "hpsdf_mesh_aabb", "hpsdf_mesh_destroy", "hpsdf_create", "hpsdf_query",
    "hpsdf_query_device", "hpsdf_query_with_gradient", "hpsdf_to_memory_block", "hpsdf_from_memory_block", "hpsdf_clone",
    "hpsdf_get_root_aabb", "hpsdf_destroy", "hpsdf_get_build_stats", "hpsdf_get_decision_log", "hpsdf_get_apply_log", "hpsdf_fit_batch",
    "hpsdf_bench_frontier", "hpsdf_measure_fp64_peak", "hpsdf_comm_get_unique_id", "hpsdf_comm_init",
    "hpsdf_comm_destroy", "hpsdf_shard_range", "hpsdf_set_jit", "hpsdf_jit_compile_check", "hpsdf_query_ray",
    "hpsdf_get_config", "hpsdf_get_device", "hpsdf_uniform_points_device", "hpsdf_extract_isosurface",
    "hpsdf_raycast", "hpsdf_raycast_device", "hpsdf_query_derivatives", "hpsdf_query_derivatives_device",
    "hpsdf_query_bounds", "hpsdf_query_bounds_device", "hpsdf_extract_isosurface_sparse",
]

_lib = None


def build_library(verbose=False):
    """Compile lib/libhpsdf.so for sm_100a (nvcc cross-compiles without a GPU)."""
    subprocess.check_call(["make", "-C", HERE, "-j8"], stdout=None if verbose else subprocess.DEVNULL)


def lib():
    """The CUDA extension. Fails loudly when it is missing: there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("%s is missing: run `make -C %s` (or __graft_entry__.build()); this package has no CPU "
                          "fallback" % (LIB_PATH, HERE))
    L = C.CDLL(LIB_PATH)
    vp, sz, dbl, u32, i32 = C.c_void_p, C.c_size_t, C.c_double, C.c_uint32, C.c_int
    L.hpsdf_status_string.restype = C.c_char_p
    L.hpsdf_status_string.argtypes = [i32]
    L.hpsdf_last_error.restype = C.c_char_p
    L.hpsdf_version.restype = C.c_char_p
    L.hpsdf_device_count.restype = i32
    L.hpsdf_config_default.argtypes = [C.POINTER(Config)]
    L.hpsdf_config_default.restype = None
    L.hpsdf_config_validate.argtypes = [C.POINTER(Config)]
    L.hpsdf_build_opts_default.argtypes = [C.POINTER(BuildOpts)]
    L.hpsdf_build_opts_default.restype = None
    L.hpsdf_sdf_eval.argtypes = [C.POINTER(_Program), vp, sz, vp, i32]
    L.hpsdf_mesh_create.argtypes = [vp, sz, vp, sz, i32, C.POINTER(vp)]
    L.hpsdf_mesh_signed_distance.argtypes = [vp, vp, sz, vp]
    L.hpsdf_mesh_aabb.argtypes = [vp, vp, vp]
    L.hpsdf_mesh_destroy.argtypes = [vp]
    L.hpsdf_mesh_destroy.restype = None
    L.hpsdf_create.argtypes = [C.POINTER(Config), C.POINTER(BuildOpts), C.POINTER(_Program), C.POINTER(vp)]
    L.hpsdf_query.argtypes = [vp, vp, sz, vp]
    L.hpsdf_query_device.argtypes = [vp, vp, sz, vp, vp]
    L.hpsdf_query_with_gradient.argtypes = [vp, vp, sz, vp, vp]
    L.hpsdf_query_ray.argtypes = [vp, vp, vp, sz, dbl, vp, vp]
    L.hpsdf_raycast.argtypes = [vp, vp, vp, sz, dbl, dbl, dbl, vp, vp]
    L.hpsdf_raycast_device.argtypes = [vp, vp, vp, sz, dbl, dbl, dbl, vp, vp, vp]
    L.hpsdf_query_derivatives.argtypes = [vp, vp, sz, vp, vp, vp]
    L.hpsdf_query_derivatives_device.argtypes = [vp, vp, sz, vp, vp, vp, vp]
    L.hpsdf_query_bounds.argtypes = [vp, vp, vp, sz, vp, vp]
    L.hpsdf_query_bounds_device.argtypes = [vp, vp, vp, sz, vp, vp, vp]
    L.hpsdf_extract_isosurface.argtypes = [vp, vp, vp, vp, dbl, C.POINTER(sz), C.POINTER(vp), C.POINTER(sz), C.POINTER(vp)]
    L.hpsdf_extract_isosurface_sparse.argtypes = L.hpsdf_extract_isosurface.argtypes
    L.hpsdf_to_memory_block.argtypes = [vp, C.POINTER(sz), C.POINTER(vp)]
    L.hpsdf_from_memory_block.argtypes = [vp, sz, i32, C.POINTER(vp)]
    L.hpsdf_clone.argtypes = [vp, C.POINTER(vp)]
    L.hpsdf_get_root_aabb.argtypes = [vp, vp, vp]
    L.hpsdf_destroy.argtypes = [vp]
    L.hpsdf_destroy.restype = None
    L.hpsdf_get_config.argtypes = [vp, C.POINTER(Config)]
    L.hpsdf_get_device.argtypes = [vp, C.POINTER(i32)]
    L.hpsdf_get_build_stats.argtypes = [vp, C.POINTER(BuildStats)]
    L.hpsdf_get_decision_log.argtypes = [vp, vp, sz]
    L.hpsdf_get_decision_log.restype = sz
    L.hpsdf_get_apply_log.argtypes = [vp, vp, sz]
    L.hpsdf_get_apply_log.restype = sz
    L.hpsdf_fit_batch.argtypes = [C.POINTER(Config), C.POINTER(_Program), vp, vp, sz, u32, vp, vp, i32, C.POINTER(C.c_float)]
    L.hpsdf_bench_frontier.argtypes = [C.POINTER(Config), C.POINTER(_Program), u32, u32, u32, i32, vp, C.POINTER(FrontierBench)]
    L.hpsdf_measure_fp64_peak.argtypes = [i32, vp, C.POINTER(dbl)]
    L.hpsdf_uniform_points_device.argtypes = [C.c_uint64, C.c_uint64, sz, C.POINTER(dbl), C.POINTER(dbl), vp, vp]
    L.hpsdf_comm_get_unique_id.argtypes = [vp]
    L.hpsdf_comm_init.argtypes = [vp, i32, i32, i32, C.POINTER(vp)]
    L.hpsdf_comm_destroy.argtypes = [vp]
    L.hpsdf_comm_destroy.restype = None
    L.hpsdf_shard_range.argtypes = [sz, i32, i32, C.POINTER(sz), C.POINTER(sz)]
    L.hpsdf_jit_compile_check.argtypes = [C.POINTER(_Program), u32, vp, sz, C.POINTER(sz)]
    L.hpsdf_set_jit.restype = None
    L.hpsdf_set_jit.argtypes = [i32]
    L.hpsdf_shard_range.restype = None
    _lib = L
    return L


def _check(status):
    if status != OK:
        raise HpsdfError(status, lib().hpsdf_last_error().decode())


def device_count():
    return lib().hpsdf_device_count()


def shard_range(n, rank, world):
    b, e = C.c_size_t(), C.c_size_t()
    lib().hpsdf_shard_range(n, rank, world, C.byref(b), C.byref(e))
    return b.value, e.value


class SdfProgram:
    """Postfix list of primitives/operators evaluated on the device; the stand-in for Create's std::function argument.

    SdfProgram([("sphere", [cx, cy, cz, r])]) ; SdfProgram([("box", [...]), ("torus", [...]), ("union", [])])
    An item may carry a handle: ("octree", [], other_octree) / ("mesh", [], mesh).
    """

    def __init__(self, items):
        self.items = list(items)
        self._instr = (Instr * len(self.items))()
        self._keep = []
        for i, it in enumerate(self.items):
            name, params = it[0], it[1]
            self._instr[i].op = PRIM[name] if name in PRIM else OP[name]
            if len(it) > 2 and it[2] is not None:
                self._keep.append(it[2])
                self._instr[i].handle = it[2]._h
            for k, v in enumerate(params):
                self._instr[i].p[k] = float(v)
        self._c = _Program(len(self.items), 0, self._instr)

    def eval(self, pts, device=-1):
        """Evaluate at user-space points on the device (test hook)."""
        pts = np.ascontiguousarray(pts, np.float64)
        out = np.empty(len(pts), np.float64)
        _check(lib().hpsdf_sdf_eval(C.byref(self._c), pts.ctypes.data, len(pts), out.ctypes.data, device))
        return out


class Mesh:
    """Device-resident triangle mesh + BVH as an SDF source (replaces Meshing::Mesh + Meshing::BVH under Create).
    verts: (n,3) float32, tris: (m,3) uint32, counter-clockwise seen from outside; raises if an edge has no twin."""

    def __init__(self, verts, tris, device=-1):
        v = np.ascontiguousarray(verts, np.float32)
        t = np.ascontiguousarray(tris, np.uint32)
        h = C.c_void_p()
        _check(lib().hpsdf_mesh_create(v.ctypes.data, len(v), t.ctypes.data, len(t), device, C.byref(h)))
        self._h = h.value

    def SignedDistanceAtPt(self, pts):
        """Mesh::SignedDistanceAtPt (Source/Meshing/Mesh.cpp:54-63), batched, float32."""
        p = np.ascontiguousarray(pts, np.float32).reshape(-1, 3)
        out = np.empty(len(p), np.float32)
        _check(lib().hpsdf_mesh_signed_distance(self._h, p.ctypes.data, len(p), out.ctypes.data))
        return out

    def CalculateMeshAABB(self):
        mn, mx = (C.c_float * 3)(), (C.c_float * 3)()
        _check(lib().hpsdf_mesh_aabb(self._h, mn, mx))
        return np.array(mn[:], np.float32), np.array(mx[:], np.float32)

    def close(self):
        if self._h:
            lib().hpsdf_mesh_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MemoryBlock:
    """MemoryBlock {size, ptr} (Include/Utility/MemoryBlock.h:5-9). `ptr` is malloc()ed by ToMemoryBlock and owned by
    the caller (the reference's callers free() it, README.md:41-53); free() here does that."""
    _libc = C.CDLL(None)
    _libc.free.argtypes = [C.c_void_p]

    def __init__(self, size, ptr, owned=True):
        self.size, self.ptr, self._owned = size, ptr, owned

    def tobytes(self):
        return C.string_at(self.ptr, self.size)

    def free(self):
        if self._owned and self.ptr:
            self._libc.free(self.ptr)
        self.ptr, self.size = None, 0

    @classmethod
    def frombytes(cls, data):
        buf = C.create_string_buffer(bytes(data), len(data))
        mb = cls(len(data), C.cast(buf, C.c_void_p).value, owned=False)
        mb._buf = buf
        return mb


class Octree:
    """SDF::Octree (Include/HP/Octree.h:36-86) on the GPU."""

    def __init__(self):
        self._h = None

    # -- Create (Octree.cpp:312-352) -----------------------------------------------------------------------------
    def Create(self, config, F, opts=None):
        """config: Config; F: SdfProgram (device SDF). Arbitrary host callables are the reference's CPU path and are
        rejected here."""
        if not isinstance(F, SdfProgram):
            raise TypeError("Create needs an SdfProgram: host lambdas stay on the reference's CPU path")
        self.Clear()
        h = C.c_void_p()
        o = opts if opts is not None else BuildOpts()
        _check(lib().hpsdf_create(C.byref(config), C.byref(o), C.byref(F._c), C.byref(h)))
        self._h = h.value
        self._keep = F

    # -- Query (Octree.cpp:662-702), batched -------------------------------------------------------------------------
    def Query(self, pts):
        """pts: (n,3) float64 (or one point) -> distances; DBL_MAX outside the root (Octree.cpp:668-671)."""
        self._need()
        a = np.ascontiguousarray(pts, np.float64)
        single = a.ndim == 1
        a = a.reshape(-1, 3)
        out = np.empty(len(a), np.float64)
        _check(lib().hpsdf_query(self._h, a.ctypes.data, len(a), out.ctypes.data))
        return float(out[0]) if single else out

    def QueryDevice(self, d_xyz_ptr, n, d_out_ptr, stream=None):
        """Device pointers (e.g. torch tensors' data_ptr()), asynchronous on `stream` (cudaStream_t as int)."""
        self._need()
        _check(lib().hpsdf_query_device(self._h, d_xyz_ptr, n, d_out_ptr, stream))

    def QueryWithGradient(self, pts):
        """Octree.cpp:749-789: (values, unit gradients)."""
        self._need()
        a = np.ascontiguousarray(pts, np.float64).reshape(-1, 3)
        out = np.empty(len(a), np.float64)
        g = np.empty((len(a), 3), np.float64)
        _check(lib().hpsdf_query_with_gradient(self._h, a.ctypes.data, len(a), out.ctypes.data, g.ctypes.data))
        return out, g

    def QueryDerivatives(self, pts, hessian=False):
        """Query's values with the exact gradients and, with hessian=True, Hessians of the hit leaves' polynomials in user
        space (hpsdf_query_derivatives, DESIGN §13) -> (values (n,), grads (n,3)[, hess (n,6): xx, xy, xz, yy, yz, zz]).
        Gradients are not normalised; outside the root the value is DBL_MAX and the derivatives are 0."""
        a = np.ascontiguousarray(pts, np.float64).reshape(-1, 3)
        v = np.empty(len(a), np.float64)
        g = np.empty((len(a), 3), np.float64)
        h = np.empty((len(a), 6), np.float64) if hessian else None
        _check(lib().hpsdf_query_derivatives(self._h, a.ctypes.data, len(a), v.ctypes.data, g.ctypes.data,
                                             h.ctypes.data if hessian else None))
        return (v, g, h) if hessian else (v, g)

    def QueryDerivativesDevice(self, d_xyz, n, d_value, d_grad, d_hess=None, stream=None):
        """QueryDerivatives with device pointers (e.g. torch tensors' data_ptr()), asynchronous on `stream` (cudaStream_t as
        int); d_hess = None skips the Hessians."""
        _check(lib().hpsdf_query_derivatives_device(self._h, d_xyz, n, d_value, d_grad, d_hess, stream))

    def QueryBounds(self, box_lo, box_hi):
        """Certified bounds of Query over closed boxes [box_lo[i], box_hi[i]] ((n,3) float64 each; hpsdf_query_bounds, DESIGN §14)
        -> (f_lo (n,), f_hi (n,)) with f_lo <= Query(x) <= f_hi for every x in box i. f_hi is DBL_MAX when part of the box is
        outside the root, both are when all of it is; a NaN or inverted box gives NaN."""
        lo = np.ascontiguousarray(box_lo, np.float64).reshape(-1, 3)
        hi = np.ascontiguousarray(box_hi, np.float64).reshape(-1, 3)
        if len(lo) != len(hi):
            raise HpsdfError(ERR_INVALID_ARG, "box_lo and box_hi differ in length")
        f_lo = np.empty(len(lo), np.float64)
        f_hi = np.empty(len(lo), np.float64)
        _check(lib().hpsdf_query_bounds(self._h, lo.ctypes.data, hi.ctypes.data, len(lo), f_lo.ctypes.data, f_hi.ctypes.data))
        return f_lo, f_hi

    def QueryBoundsDevice(self, d_lo, d_hi, n, d_flo, d_fhi, stream=None):
        """QueryBounds with device pointers (e.g. torch tensors' data_ptr()), asynchronous on `stream` (cudaStream_t as int)."""
        _check(lib().hpsdf_query_bounds_device(self._h, d_lo, d_hi, n, d_flo, d_fhi, stream))

    def QueryTorch(self, x):
        """Query as a differentiable torch function: x is a contiguous CUDA float64 (n,3) tensor on the tree's device, the
        result (n,) float64, computed on the current stream of that device. Autograd gets the exact gradient from the
        forward launch, and the exact Hessian on a second differentiation (create_graph=True); a third raises. Nothing is
        copied: another dtype, device, shape or layout raises."""
        import torch
        self._need()
        if not isinstance(x, torch.Tensor) or x.dtype != torch.float64:
            raise TypeError("QueryTorch needs a float64 torch tensor")
        dev = C.c_int()
        _check(lib().hpsdf_get_device(self._h, C.byref(dev)))
        if x.device.type != "cuda" or x.device.index != dev.value:
            raise ValueError("QueryTorch needs a tensor on cuda:%d, the tree's device (got %s)" % (dev.value, x.device))
        if x.dim() != 2 or x.shape[1] != 3 or not x.is_contiguous():
            raise ValueError("QueryTorch needs a contiguous (n, 3) tensor (got shape %s)" % (tuple(x.shape),))
        if x.requires_grad and torch.is_grad_enabled():
            return _torch_query()[0].apply(x, self)
        return _torch_launch(self, x, 0)[0]

    def QueryRay(self, origins, directions, t_max):
        """Octree::QueryRay (Octree.cpp:705-746) for a batch of rays -> (hit flags, t). Mirrors the reference statement by statement."""
        self._need()
        o = np.ascontiguousarray(origins, np.float64).reshape(-1, 3)
        d = np.ascontiguousarray(directions, np.float64).reshape(-1, 3)
        assert len(o) == len(d)
        hit = np.zeros(len(o), np.uint8)
        t = np.zeros(len(o), np.float64)
        _check(lib().hpsdf_query_ray(self._h, o.ctypes.data, d.ctypes.data, len(o), float(t_max), hit.ctypes.data, t.ctypes.data))
        return hit.astype(bool), t

    def Raycast(self, origins, directions, t_min=0.0, t_max=np.inf, iso=0.0):
        """First crossing of F = iso along rays o + t d, t in [t_min, t_max] (hpsdf_raycast; d need not be unit, t is in units
        of d) -> (t (n,) f64, +inf for a miss; normals (n,3) f64, unit gradients of the hit leaf's polynomial, 0 on a miss).
        Exact per leaf (DESIGN §12); the ray query to use, where QueryRay mirrors the reference."""
        o = np.ascontiguousarray(origins, np.float64).reshape(-1, 3)
        d = np.ascontiguousarray(directions, np.float64).reshape(-1, 3)
        if len(o) != len(d):
            raise HpsdfError(ERR_INVALID_ARG, "origins and directions differ in length")
        t = np.empty(len(o), np.float64)
        nrm = np.empty((len(o), 3), np.float64)
        _check(lib().hpsdf_raycast(self._h, o.ctypes.data, d.ctypes.data, len(o), float(t_min), float(t_max), float(iso),
                                   t.ctypes.data, nrm.ctypes.data))
        return t, nrm

    def RaycastDevice(self, d_origins, d_directions, n, d_t, d_normals=None, t_min=0.0, t_max=np.inf, iso=0.0, stream=None):
        """Raycast with device pointers (e.g. torch tensors' data_ptr()), asynchronous on `stream` (cudaStream_t as int)."""
        _check(lib().hpsdf_raycast_device(self._h, d_origins, d_directions, n, float(t_min), float(t_max), float(iso), d_t, d_normals,
                                          stream))

    def OutputFunctionSlice(self, fname, c, view_min, view_max, n_samples=2048):
        """Octree::OutputFunctionSlice (Octree.cpp:1132-1205): the z = c slice of the field over viewArea as an n x n grid of
        batched Queries (the reference loops 2048^2 scalar Queries), coloured like the reference (green outside, blue inside,
        each rescaled to its own range) and written as `fname`.bmp when fname is not None. Returns (values, rgb image).
        Sample positions use the reference's arithmetic: one float32 step from the x extent for both axes (:1150-1153)."""
        self._need()
        vmin = np.asarray(view_min, np.float32)
        vmax = np.asarray(view_max, np.float32)
        n = int(n_samples)
        step = np.float32((vmax[0] - vmin[0]) / np.float32(n))
        idx = np.arange(n, dtype=np.uint32).astype(np.float32)
        xs = vmin[0].astype(np.float64) + (idx * step).astype(np.float64)
        ys = vmin[1].astype(np.float64) + (idx * step).astype(np.float64)
        pts = np.empty((n, n, 3), np.float64)
        pts[:, :, 0] = xs[None, :]
        pts[:, :, 1] = ys[:, None]
        pts[:, :, 2] = float(c)
        vals = self.Query(pts.reshape(-1, 3)).reshape(n, n)
        eps = np.float64(np.float32(0.000001))
        pos, v32 = vals > eps, vals.astype(np.float32)
        pmin, pmax = (vals[pos].min(), vals[pos].max()) if pos.any() else (np.finfo(np.float64).max, 0.0)
        nmin, nmax = (vals[~pos].min(), vals[~pos].max()) if (~pos).any() else (0.0, -np.finfo(np.float64).max)
        img = np.zeros((n, n, 3), np.uint8)
        with np.errstate(divide="ignore", invalid="ignore"):
            g = 255 * (v32.astype(np.float64) - pmax) / (pmin - pmax)
            b = 255 * (v32.astype(np.float64) - nmin) / (nmax - nmin)
        outside = v32 > 0.0
        img[:, :, 1] = np.where(outside, np.nan_to_num(g, nan=0.0, posinf=255.0, neginf=0.0).clip(0, 255), 0).astype(np.uint8)
        img[:, :, 2] = np.where(~outside, np.nan_to_num(b, nan=0.0, posinf=255.0, neginf=0.0).clip(0, 255), 0).astype(np.uint8)
        if fname is not None:
            row = (3 * n + 3) & ~3
            hdr = b"BM" + (54 + row * n).to_bytes(4, "little") + bytes(4) + (54).to_bytes(4, "little") + (40).to_bytes(4, "little") + \
                n.to_bytes(4, "little") + n.to_bytes(4, "little") + (1).to_bytes(2, "little") + (24).to_bytes(2, "little") + bytes(24)
            with open(str(fname) + ".bmp", "wb") as f:
                f.write(hdr)
                pad = bytes(row - 3 * n)
                for i in range(n - 1, -1, -1):                      # BMP rows are stored bottom-up; channels as B, G, R
                    f.write(img[i, :, ::-1].tobytes() + pad)
        return vals, img

    def ExtractIsosurface(self, resolution, iso=0.0, box=None):
        """The level set F = iso as a triangle mesh (hpsdf_extract_isosurface): marching tetrahedra over a uniform grid of
        `resolution` cells per axis (an int or 3 ints, each 1..1024) spanning box = (min xyz, max xyz), or the root box.
        Returns (vertices (n,3) float32, triangles (m,3) uint32), counter-clockwise seen from the side where F >= iso; closed
        when the surface stays inside the box. hp.Mesh(vertices, triangles) takes it as it is."""
        return self._extract(lib().hpsdf_extract_isosurface, 1024, resolution, iso, box)

    def ExtractIsosurfaceSparse(self, resolution, iso=0.0, box=None):
        """ExtractIsosurface's mesh, bit for bit, on grids of up to 16384 cells per axis (hpsdf_extract_isosurface_sparse,
        DESIGN §15): only the blocks of 16^3 cells whose certified bounds (QueryBounds) reach iso are evaluated, so the work
        and device memory grow with the surface, not with the grid."""
        return self._extract(lib().hpsdf_extract_isosurface_sparse, 16384, resolution, iso, box)

    def _extract(self, fn, limit, resolution, iso, box):
        res = [int(resolution)] * 3 if np.ndim(resolution) == 0 else [int(r) for r in resolution]
        if len(res) != 3 or not all(0 <= r <= 0xFFFFFFFF for r in res):
            raise HpsdfError(ERR_INVALID_ARG, "resolution must be one or three counts in [1, %d]" % limit)
        lo = hi = None
        if box is not None:
            lo, hi = ((C.c_double * 3)(*[float(x) for x in b]) for b in box)
        nv, nt, pv, pt = C.c_size_t(), C.c_size_t(), C.c_void_p(), C.c_void_p()
        _check(fn(self._h, (C.c_uint32 * 3)(*res), lo, hi, float(iso), C.byref(nv), C.byref(pv), C.byref(nt), C.byref(pt)))
        try:
            v = np.ctypeslib.as_array((C.c_float * (3 * nv.value)).from_address(pv.value)).reshape(-1, 3).copy() if nv.value else np.empty((0, 3), np.float32)
            t = np.ctypeslib.as_array((C.c_uint32 * (3 * nt.value)).from_address(pt.value)).reshape(-1, 3).copy() if nt.value else np.empty((0, 3), np.uint32)
        finally:
            MemoryBlock._libc.free(pv)
            MemoryBlock._libc.free(pt)
        return v, t

    # -- serialisation (Octree.cpp:403-456) ----------------------------------------------------------------------------
    def ToMemoryBlock(self):
        self._need()
        size, ptr = C.c_size_t(), C.c_void_p()
        _check(lib().hpsdf_to_memory_block(self._h, C.byref(size), C.byref(ptr)))
        return MemoryBlock(size.value, ptr.value)

    def FromMemoryBlock(self, block, device=-1):
        """Copies; the caller keeps ownership of the block (HPUnitTests.cpp:136-138)."""
        self.Clear()
        h = C.c_void_p()
        _check(lib().hpsdf_from_memory_block(block.ptr, block.size, device, C.byref(h)))
        self._h = h.value

    def Clear(self):
        if self._h:
            lib().hpsdf_destroy(self._h)
        self._h = None

    def copy(self):
        """Copy constructor (Octree.cpp:24-45)."""
        self._need()
        h = C.c_void_p()
        _check(lib().hpsdf_clone(self._h, C.byref(h)))
        o = Octree()
        o._h = h.value
        return o

    def GetRootAABB(self):
        self._need()
        mn, mx = (C.c_float * 3)(), (C.c_float * 3)()
        _check(lib().hpsdf_get_root_aabb(self._h, mn, mx))
        return np.array(mn[:], np.float32), np.array(mx[:], np.float32)

    # -- SDF boolean operations (Octree.cpp:355-400): re-Create from min/max of the old tree's Query and F ----------------
    def _combine(self, F, op, opts=None):
        """opts (BuildOpts) carries max_degree / max_depth / ...; the rebuild runs on the old tree's device unless opts.device
        names one. A failed rebuild leaves the tree as it was."""
        self._need()
        old = Octree()
        old._h, self._h = self._h, None
        try:
            cfg = Config()
            _check(lib().hpsdf_get_config(old._h, C.byref(cfg)))
            o = BuildOpts()
            if opts is not None:
                C.memmove(C.byref(o), C.byref(opts), C.sizeof(BuildOpts))
            if o.device < 0:
                dev = C.c_int()
                _check(lib().hpsdf_get_device(old._h, C.byref(dev)))
                o.device = dev.value
            prog = SdfProgram(list(F.items) + [("octree", [], old), (op, [])])
            self.Create(cfg, prog, o)
        except Exception:
            self.Clear()
            self._h, old._h = old._h, None
            raise
        old.Clear()

    def UnionSDF(self, F, opts=None):
        self._combine(F, "union", opts)           # min(oldF, F)

    def IntersectSDF(self, F, opts=None):
        self._combine(F, "intersect", opts)       # max(oldF, F)

    def SubtractSDF(self, F, opts=None):
        self._combine(F, "subtract", opts)        # max(F, -oldF)

    # -- extras ------------------------------------------------------------------------------------------------------
    def ToMemoryBlockBytes(self):
        mb = self.ToMemoryBlock()
        try:
            return mb.tobytes()
        finally:
            mb.free()

    def stats(self):
        self._need()
        s = BuildStats()
        _check(lib().hpsdf_get_build_stats(self._h, C.byref(s)))
        return s.as_dict()

    def decision_log(self):
        self._need()
        n = lib().hpsdf_get_decision_log(self._h, None, 0)
        arr = (DecisionLogEntry * max(n, 1))()
        lib().hpsdf_get_decision_log(self._h, arr, n)
        return [dict(node_idx=e.node_idx, depth=e.depth, degree=e.degree, centre=tuple(e.centre), chose_p=e.chose_p,
                     kind=e.kind, p_improvement=e.p_improvement, h_improvement=e.h_improvement,
                     relative_margin=e.relative_margin) for e in arr[:n]]

    def apply_log(self):
        """(n, 8) array: node, kind (0 P / 1 H), degree, initial_err, new_err, p_imp, h_imp, total_after — the same
        columns the CPU checker's apply log has."""
        self._need()
        n = lib().hpsdf_get_apply_log(self._h, None, 0)
        arr = (ApplyLogEntry * max(n, 1))()
        lib().hpsdf_get_apply_log(self._h, arr, n)
        return np.array([[e.node_idx, e.kind, e.degree, e.initial_err, e.new_err, e.p_improvement, e.h_improvement,
                          e.total_after] for e in arr[:n]], np.float64).reshape(n, 8)

    def _need(self):
        if not self._h:
            raise HpsdfError(ERR_INVALID_ARG, "octree is empty (call Create or FromMemoryBlock)")

    def __del__(self):
        try:
            self.Clear()
        except Exception:
            pass


def _torch_launch(tree, x, order):
    """Query (order 0) or the derivatives (order 1, 2) of a checked CUDA tensor x, on the current stream of its device."""
    import torch
    n = x.shape[0]
    v = torch.empty(n, dtype=torch.float64, device=x.device)
    g = torch.empty((n, 3), dtype=torch.float64, device=x.device) if order >= 1 else None
    h = torch.empty((n, 6), dtype=torch.float64, device=x.device) if order == 2 else None
    with torch.cuda.device(x.device):
        stream = torch.cuda.current_stream(x.device).cuda_stream
        if order == 0:
            _check(lib().hpsdf_query_device(tree._h, x.data_ptr(), n, v.data_ptr(), stream))
        else:
            _check(lib().hpsdf_query_derivatives_device(tree._h, x.data_ptr(), n, v.data_ptr(), g.data_ptr(),
                                                        h.data_ptr() if h is not None else None, stream))
    return v, g, h


_TORCH_QUERY = None


def _torch_query():
    """The autograd functions behind Octree.QueryTorch, defined on first use so that importing this package needs no torch."""
    global _TORCH_QUERY
    if _TORCH_QUERY is not None:
        return _TORCH_QUERY
    import torch

    class QueryFn(torch.autograd.Function):
        """F(x): one ORDER-1 launch gives the value and keeps the gradient for backward."""

        @staticmethod
        def forward(ctx, x, tree):
            v, g, _ = _torch_launch(tree, x, 1)
            ctx.tree = tree
            ctx.save_for_backward(x, g)
            return v

        @staticmethod
        def backward(ctx, gv):
            x, g = ctx.saved_tensors
            return GradFn.apply(x, gv, g, ctx.tree), None

    class GradFn(torch.autograd.Function):
        """gv[:, None] * grad F(x); its backward is the Hessian-vector product from one ORDER-2 launch."""

        @staticmethod
        def forward(ctx, x, gv, g, tree):
            ctx.tree = tree
            ctx.save_for_backward(x, gv, g)
            return gv[:, None] * g

        @staticmethod
        def backward(ctx, w):
            x, gv, g = ctx.saved_tensors
            gx = ggv = None
            if ctx.needs_input_grad[0]:
                H = _torch_launch(ctx.tree, x.detach(), 2)[2]
                Hw = torch.stack([H[:, 0] * w[:, 0] + H[:, 1] * w[:, 1] + H[:, 2] * w[:, 2],
                                  H[:, 1] * w[:, 0] + H[:, 3] * w[:, 1] + H[:, 4] * w[:, 2],
                                  H[:, 2] * w[:, 0] + H[:, 4] * w[:, 1] + H[:, 5] * w[:, 2]], 1)
                gx = gv[:, None] * Hw
            if ctx.needs_input_grad[1]:
                ggv = (g * w).sum(1)
            if torch.is_grad_enabled():
                gx, ggv = NoThirdOrder.apply(x, gx, ggv)
            return gx, ggv, None, None

    class NoThirdOrder(torch.autograd.Function):
        """Passes the second derivatives through; differentiating them (a third derivative of F) raises."""

        @staticmethod
        def forward(ctx, x, gx, ggv):
            return (None if gx is None else gx.clone()), (None if ggv is None else ggv.clone())

        @staticmethod
        def backward(ctx, *_):
            raise RuntimeError("Octree.QueryTorch is differentiable twice: a third derivative of the field is not available")

    _TORCH_QUERY = (QueryFn, GradFn)
    return _TORCH_QUERY


def fit_batch(config, F, cells, depth, degree, device=-1):
    """FitPolynomial (Octree.cpp:1007-1093) for independent cells, from scratch. cells: (n,4) f32 {cx,cy,cz,half}."""
    cells = np.ascontiguousarray(cells, np.float32)
    depth = np.ascontiguousarray(depth, np.uint8)
    n = len(cells)
    coeffs = np.empty((n, COEFF_COUNT[degree]), np.float64)
    err = np.empty(n, np.float64)
    ms = C.c_float()
    _check(lib().hpsdf_fit_batch(C.byref(config), C.byref(F._c), cells.ctypes.data, depth.ctypes.data, n, degree,
                                 coeffs.ctypes.data, err.ctypes.data, device, C.byref(ms)))
    return coeffs, err, ms.value


def bench_frontier(config, F, grid_depth, degree, repeats=3, device=-1, stream=None):
    out = FrontierBench()
    _check(lib().hpsdf_bench_frontier(C.byref(config), C.byref(F._c), grid_depth, degree, repeats, device, stream, C.byref(out)))
    return {k: getattr(out, k) for k, _ in out._fields_}


def set_jit(on):
    """Process default for BuildOpts.jit == 0, fit_batch and bench_frontier: NVRTC-specialised fit kernels for closed-form programs."""
    lib().hpsdf_set_jit(1 if on else 0)


def jit_compile_check(F, degree):
    """Generate + NVRTC-compile the specialised fit kernel of `degree` for program F (no GPU needed) -> (source, cubin bytes)."""
    buf = C.create_string_buffer(1 << 16)
    n = C.c_size_t()
    _check(lib().hpsdf_jit_compile_check(C.byref(F._c), degree, buf, len(buf), C.byref(n)))
    return buf.value.decode(), n.value


def uniform_points_device(seed, first_index, n, lo, hi, d_xyz_ptr, stream=None):
    """Philox4x32-10 points (key = seed, counter = global point index) uniform in [lo, hi) into a device buffer of n x 3 f64."""
    _check(lib().hpsdf_uniform_points_device(seed, first_index, n, (C.c_double * 3)(*[float(v) for v in lo]),
                                             (C.c_double * 3)(*[float(v) for v in hi]), d_xyz_ptr, stream))


def measure_fp64_peak(device=-1, stream=None):
    t = C.c_double()
    _check(lib().hpsdf_measure_fp64_peak(device, stream, C.byref(t)))
    return t.value


def parse_block(block):
    """MemoryBlock bytes (LP64 layout, SURVEY.md App. B) -> dict of numpy views; compare field-wise, never memcmp."""
    b = np.frombuffer(bytes(block), dtype=np.uint8)
    ncoef = int(b[:8].view(np.uint64)[0])
    coeffs = b[8:8 + 8 * ncoef].view(np.float64)
    off = 8 + 8 * ncoef
    nnodes = int(b[off:off + 8].view(np.uint64)[0])
    off += 8
    node_dt = np.dtype({"names": ["child", "mn", "mx", "cstart", "deg", "depth"],
                        "formats": ["<u8", ("<f4", 3), ("<f4", 3), "<u8", "u1", "u1"],
                        "offsets": [0, 8, 20, 32, 40, 48], "itemsize": 56})
    nodes = b[off:off + 56 * nnodes].view(node_dt)
    off += 56 * nnodes
    if off + 80 != len(b):
        raise ValueError("block size mismatch")
    cfg = Config.from_buffer_copy(bytes(b[off:off + 80]))
    return dict(n_coeffs=ncoef, coeffs=coeffs, n_nodes=nnodes, nodes=nodes, config=cfg)


class Comm:
    """One rank of a multi-GPU build (NCCL). Rank 0 makes the id; ship it with torch.distributed / any transport."""

    def __init__(self, unique_id, rank, world, device):
        h = C.c_void_p()
        buf = C.create_string_buffer(bytes(unique_id), 128)
        _check(lib().hpsdf_comm_init(buf, rank, world, device, C.byref(h)))
        self._h, self.rank, self.world = h.value, rank, world

    @staticmethod
    def unique_id():
        buf = C.create_string_buffer(128)
        _check(lib().hpsdf_comm_get_unique_id(buf))
        return buf.raw

    def close(self):
        if self._h:
            lib().hpsdf_comm_destroy(self._h)
            self._h = None
