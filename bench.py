#!/usr/bin/env python
"""bench.py — the reference's headline metric on B200: octree build nodes-fitted/s (+ Query points/s) vs CPU.

    python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (CUDA through the C ABI)
    python bench.py ... --dump-outputs DIR                         + the headline tree of the last timed step as DIR/*.npy
    python bench.py --impl reference [--steps K] [--warmup W]      the reference's own CPU implementation (oracle/_ref)
    torchrun --nproc-per-node N ... bench.py --gpus N ...          N > 1: one rank per GPU (NCCL)

Headline workload = BASELINE.json configs[2] ("c3_dragon_standin": mesh SDF over a GPU BVH with pseudonormals, threshold
1e-6, continuity strength 8) on the 870 000-triangle procedural stand-in of the absent dragon.obj (SURVEY.md §8d): the
largest configuration that fits one GPU AND has a feasible stock-reference arm (one Octree::Create of it takes the
reference ~1 minute on 16 host cores; configs[3] would take hours). A "step" is one Octree::Create of it; with N > 1 the
ranks build ONE tree together (frontier sharded, NCCL exchange per round): strong scaling.
`value` = nodes fitted per second: FitPolynomial-equivalents on the strict-greedy path (4096 coarse fits + 9 per applied
refinement job — a constant of the workload, tests/golden/workloads.json) / time of the Create, mesh and BVH already
resident in HBM. `e2e` goes through the public API from HOST buffers: vertex / index arrays in, hpsdf_mesh_create (upload +
half-edges + pseudonormals + BVH), Create, ToMemoryBlock out, all inside the timed region.

Sub-objects of the same JSON line (each with its own CPU figure at N = 1): `c1_readme` (README sphere, continuity),
`c2_csg` (closed-form CSG build with NVRTC-specialised fit kernels + the fit-kernel FP64 roofline on the synthetic
frontier), `c4_ramesses_standin` (1.6 M triangles, threshold 1e-8, max degree 6), `c5_query_1e9` (10^9 Philox points on the
C3 tree, replicated tree, points sharded) and `query` (2^24-point launches: the HBM roofline of queryKernel).

Prints ONE JSON line on rank 0.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from cases import CASES, leaf_table, path_code  # noqa: E402

PKG = "hp-adaptive-signed-distance-field-octree_b200"
WORKLOAD = "c3_dragon_standin"
METRIC = "octree_build_nodes_fitted_per_s"
QUERY_POINTS = 1 << 24            # 16.7 M points = 512 MB in + 128 MB out: larger than the 126 MB L2
NCU_QUERY_TRAFFIC_BYTES = 405746176 + 119461632
MESH_UV = (1000, 435)             # bumpy torus with 870 000 triangles: the stand-in of configs[2]'s dragon.obj (absent from the reference tree)
MESH_C4_UV = (1000, 800)          # 1.6 M triangles: the stand-in of configs[3]'s Ramesses.obj
C3 = dict(threshold=1e-6, continuity=True, cstrength=8.0, max_degree=11)
C4 = dict(threshold=1e-8, continuity=False, cstrength=8.0, max_degree=6)
SEED = 0x5DF0C7EE
if os.environ.get("HPSDF_BENCH_DEV_SMALL"):      # development only: tiny meshes so the legs can be exercised quickly; the line says so
    MESH_UV, MESH_C4_UV, WORKLOAD = (120, 60), (160, 80), "c3_dragon_standin_DEV_SMALL_NOT_A_RESULT"
NOCHILD = np.uint64(0xFFFFFFFFFFFFFFFF)


def workload_constants():
    p = os.path.join(ROOT, "tests", "golden", "workloads.json")
    return json.load(open(p)) if os.path.exists(p) else {}


def headline_config():
    """The `config` object of the JSON line: the same dict from both arms."""
    w = workload_constants().get(WORKLOAD, {})
    return {"workload": WORKLOAD, "sdf": "triangle mesh, bumpy torus U=%d V=%d (stand-in of dragon.obj)" % MESH_UV,
            "triangles": 2 * MESH_UV[0] * MESH_UV[1], "threshold": C3["threshold"], "continuity_strength": C3["cstrength"],
            "root": "mesh AABB centre +- 0.6 max extent", "nodes_fitted_per_step": w.get("nodes_fitted"),
            "n_nodes": w.get("n_nodes"), "n_coeffs": w.get("n_coeffs"),
            "l2": "a 256 MB buffer is overwritten between timed steps (GPU arm); the mesh + BVH (120 MB) and 109 MB of samples per build exceed L2 anyway"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d.get("hbm_gbs", 6650.0)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.rows, self.stop, self.index = [], False, index
        self.th = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.th.join(timeout=6)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def product_case(hp, name):
    k = CASES[name]["cfg"]
    cfg = hp.Config(target_error_threshold=k["threshold"], nearness_type=k.get("nearness", 0),
                    nearness_strength=k.get("strength", 0.0), continuity_enforce=1 if k.get("continuity", True) else 0,
                    continuity_strength=k.get("cstrength", 8.0), thread_count=os.cpu_count() or 1,
                    root_min=k.get("root_min", (-0.5,) * 3), root_max=k.get("root_max", (0.5,) * 3))
    return cfg, hp.SdfProgram(CASES[name]["prog"])


def useful_fits(stats):
    """FitPolynomial-equivalents on the strict-greedy path: 4096 coarse fits + the 9 fits of every applied job."""
    return 4096 + 9 * (stats["jobs_applied_p"] - 4096 + stats["jobs_applied_h"])


def canonical_equal(hp, raw_a, raw_b):
    """Bit-equality of two MemoryBlocks up to node numbering: same leaves (path, depth, degree) with identical coefficients."""
    a, b = hp.parse_block(raw_a), hp.parse_block(raw_b)
    if a["n_nodes"] != b["n_nodes"] or a["n_coeffs"] != b["n_coeffs"]:
        return False
    pa, da, ga, ca = leaf_table(a, hp.COEFF_COUNT)
    pb, db, gb, cb = leaf_table(b, hp.COEFF_COUNT)
    return pa == pb and np.array_equal(da, db) and np.array_equal(ga, gb) and all(np.array_equal(x, y) for x, y in zip(ca, cb))


class Ctx:
    """What every leg needs: torch, the package, rank layout, the build stream, the library communicator."""

    def __init__(self):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.hp = importlib.import_module(PKG)
        self.dist, self.comm = None, None
        if self.world > 1:
            import torch.distributed as dist
            self.dist = dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            uid = torch.zeros(128, dtype=torch.uint8, device="cuda")          # NCCL id of the library's own communicator
            if self.rank == 0:
                uid.copy_(torch.frombuffer(bytearray(self.hp.Comm.unique_id()), dtype=torch.uint8))
            dist.broadcast(uid, 0)
            self.comm = self.hp.Comm(bytes(uid.cpu().numpy().tobytes()), self.rank, self.world, self.local)
        self.stream = torch.cuda.current_stream().cuda_stream
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, *xs):
        t = self.torch.tensor(list(xs), dtype=self.torch.float64, device="cuda")
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t.cpu()]

    def opts(self, sharded=True, **kw):
        o = self.hp.BuildOpts(device=self.local, stream=self.stream, **kw)
        if sharded and self.comm is not None:
            o.comm = self.comm._h
        return o

    def timed_creates(self, tree, cfg, prog, opts, steps, warmup):
        """W untimed + K timed Creates, each bracketed by CUDA events on the build stream, L2 overwritten in between.
        Returns (ms per step: max over ranks of the device time, or of the wall time when ranks cooperate; stats sums)."""
        torch = self.torch
        for _ in range(warmup):
            tree.Create(cfg, prog, opts)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        agg = {}
        self.barrier()
        wall = 0.0
        for i in range(steps):
            self.flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ev[i][0].record()
            tree.Create(cfg, prog, opts)
            ev[i][1].record()
            torch.cuda.synchronize()
            wall += time.perf_counter() - t0
            for k, v in tree.stats().items():
                agg[k] = agg.get(k, 0) + v
        self.barrier()
        dev_ms = sum(a.elapsed_time(b) for a, b in ev)
        dev_ms, wall_ms = self.max_over_ranks(dev_ms, 1e3 * wall)
        ms = (max(dev_ms, wall_ms) if self.world > 1 else dev_ms) / steps
        return ms, agg


def mesh_case(cx, uv, spec):
    from meshgen import bumpy_torus, mesh_root
    hp = cx.hp
    verts, tris = bumpy_torus(*uv)
    mn, mx = mesh_root(verts)
    cfg = hp.Config(target_error_threshold=spec["threshold"], nearness_type=0, nearness_strength=0.0,
                    continuity_enforce=1 if spec["continuity"] else 0, continuity_strength=spec["cstrength"],
                    thread_count=os.cpu_count() or 1, root_min=mn, root_max=mx)
    return verts, tris, (mn, mx), cfg


def cpu_fit_sample(hp, tree, verts, tris, box, spec, budget_s=15.0):
    """The reference's FitPolynomial over the reference's Mesh + BVH (oracle/_ref, -O3 + OpenMP build) on a bounded random
    sample of the refinement jobs this very build applied (8 child fits + 1 kept-shell fit each), all host threads."""
    from oracle import hpref
    if not hpref.available(fast=True):
        return {"unavailable": "oracle/_ref/libhpref_fast.so not built"}
    threads = os.cpu_count() or 1
    t0 = time.perf_counter()
    rm = hpref.RefMesh.create(verts, tris, True, fast=True)
    setup_s = time.perf_counter() - t0
    rcfg = hpref.make_config(threshold=spec["threshold"], continuity=False, root_min=box[0], root_max=box[1], threads=threads)
    rprog = hpref.make_program([("mesh", [], rm.h)])
    blk = hp.parse_block(tree.ToMemoryBlockBytes())
    nodes = blk["nodes"]
    log = tree.apply_log()
    jobs = log[(log[:, 2] >= 2)]                          # refinement jobs (the 4096 coarse fits have degree 0)
    rng = np.random.default_rng(7)

    def fit_list(rows):
        mn, mx, d0, d1, dep, kept = [], [], [], [], [], []
        for r in rows:
            i, p = int(r[0]), int(r[2])
            lo, hi, depth = nodes["mn"][i].astype(np.float32), nodes["mx"][i].astype(np.float32), int(nodes["depth"][i])
            mid = (lo + hi) * np.float32(0.5)
            if depth < 10:
                for c in range(8):
                    sel = np.array([(c >> a) & 1 for a in range(3)], bool)
                    mn.append(np.where(sel, mid, lo)); mx.append(np.where(sel, hi, mid)); d0.append(p); d1.append(p); dep.append(depth + 1); kept.append(0)
            if p < spec["max_degree"]:
                mn.append(lo); mx.append(hi); d0.append(p + 1); d1.append(p + 1); dep.append(depth); kept.append(p)
        return mn, mx, d0, d1, dep, kept

    def run(rows):
        mn, mx, d0, d1, dep, kept = fit_list(rows)
        t0 = time.perf_counter()
        hpref.ref_fit_chain_batch(rcfg, rprog, np.array(mn), np.array(mx), d0, d1, dep, threads=threads, fast=True, kept_degree=kept)
        return len(mn), time.perf_counter() - t0

    pilot = jobs[rng.choice(len(jobs), min(2 * threads, len(jobs)), replace=False)]
    n0, s0 = run(pilot)
    more = int(min(len(jobs), max(2 * threads, len(pilot) * (budget_s - s0) / max(s0, 1e-3))))
    rows = jobs[rng.choice(len(jobs), more, replace=False)]
    n1, s1 = run(rows)
    return {"value": n1 / s1, "unit": "fits/s", "cores": threads, "kind": "reference",
            "sample": "%d of the %d refinement jobs this build applied (%d FitPolynomial calls: 8 child fits + 1 kept-shell fit per job) "
                      "through the reference's FitPolynomial + Mesh::SignedDistanceAtPt + BVH, OpenMP over fits, %.1f s"
                      % (len(rows), len(jobs), n1, s1),
            "reference_mesh_and_bvh_setup_s": setup_s}


def bench_c3(cx, args, clk_holder):
    """Headline: configs[2] stand-in. Returns (line fields, tree, host arrays for the later legs)."""
    hp, torch = cx.hp, cx.torch
    verts, tris, box, cfg = mesh_case(cx, MESH_UV, C3)
    t0 = time.perf_counter()
    mesh = hp.Mesh(verts, tris, device=cx.local)
    mesh_setup_s = time.perf_counter() - t0
    prog = hp.SdfProgram([("mesh", [], mesh)])
    opts = cx.opts(max_degree=C3["max_degree"])
    tree = hp.Octree()
    with ClockSampler(cx.local) as clk:
        ms, agg = cx.timed_creates(tree, cfg, prog, opts, args.steps, args.warmup)
    clk_holder.append(clk.summary())
    st = tree.stats()
    fits = useful_fits(st)
    out = {"ms_per_step": ms, "fits": fits, "stats": st, "agg": agg, "mesh_setup_s": mesh_setup_s}

    # cooperative build == solo build, bit for bit (canonical tree, coefficients, Query), checked on rank 0 in this very run
    if cx.world > 1:
        ok = None
        if cx.rank == 0:
            solo = hp.Octree()
            solo.Create(cfg, prog, cx.opts(sharded=False, max_degree=C3["max_degree"]))
            pts = np.random.default_rng(3).uniform(box[0], box[1], (200000, 3))
            ok = bool(canonical_equal(hp, tree.ToMemoryBlockBytes(), solo.ToMemoryBlockBytes()) and np.array_equal(tree.Query(pts), solo.Query(pts)))
            solo.Clear()
        cx.barrier()
        out["multi_gpu_parity"] = ok

    # e2e: host arrays (pinned, as the contract asks) -> mesh set-up -> Create -> MemoryBlock on the host, every step
    pv = torch.from_numpy(np.ascontiguousarray(verts, np.float32)).pin_memory()
    pt = torch.from_numpy(np.ascontiguousarray(tris, np.uint32).view(np.int32)).pin_memory()
    verts_p, tris_p = pv.numpy(), pt.numpy().view(np.uint32)
    n_e2e = max(2, min(args.steps, 5))
    cx.barrier()
    times, blk_bytes = [], 0
    for i in range(n_e2e + 1):
        t0 = time.perf_counter()
        m2 = hp.Mesh(verts_p, tris_p, device=cx.local)
        t2 = hp.Octree()
        t2.Create(cfg, hp.SdfProgram([("mesh", [], m2)]), opts)
        blk = t2.ToMemoryBlock()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
        blk_bytes = blk.size
        blk.free()
        t2.Clear()
        m2.close()
        if cx.dist is not None:
            cx.dist.barrier()
    e2e_ms = cx.max_over_ranks(1e3 * float(np.mean(times[1:])))[0]
    out["e2e"] = {"value": fits / (e2e_ms * 1e-3), "unit": "fits/s", "ms_per_step": e2e_ms, "steps": n_e2e,
                  "h2d_bytes_per_step": int(verts.nbytes + tris.nbytes + 160 + 32 * st["jobs_evaluated"]),
                  "d2h_bytes_per_step": int(blk_bytes + 16 * st["fits_evaluated"]),
                  "what": "hpsdf_mesh_create from host vertex / index arrays + hpsdf_create + hpsdf_to_memory_block, per step"}
    return out, tree, mesh, verts, tris, box, cfg


def dump_outputs(hp, tree, out_dir):
    """The tree of the last timed Create as its caller reads it back (ToMemoryBlock), leaves in canonical order (depth first
    by child slot), so that two builds compare array for array even where they number their nodes differently. The headline
    tree holds about 0.8 MB of coefficients."""
    paths, depth, deg, cs = leaf_table(hp.parse_block(tree.ToMemoryBlockBytes()), hp.COEFF_COUNT)
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"leaf_code": np.array([path_code(p) for p in paths], np.float64),       # 3 bits per level: exact in float64
              "leaf_depth": depth.astype(np.float64), "leaf_degree": deg.astype(np.float64),
              "leaf_coeffs": np.concatenate(cs).astype(np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def bench_c5(cx, tree, box):
    """configs[4]: 1e9 Philox points (key = seed, counter = global point index) on the C3 octree, replicated tree, points sharded
    contiguously, generated on the device in chunks of 2^26 (untimed); every N evaluates the same point set."""
    hp, torch = cx.hp, cx.torch
    total, chunk = 1_000_000_000, 1 << 26
    b, e = hp.shard_range(total, cx.rank, cx.world)
    pts = torch.empty((chunk, 3), device="cuda", dtype=torch.float64)
    out = torch.empty(chunk, device="cuda", dtype=torch.float64)
    q_ms, done = 0.0, b
    bits = torch.zeros(1, dtype=torch.int64, device="cuda")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cx.barrier()
    while done < e:
        m = min(chunk, e - done)
        hp.uniform_points_device(SEED, done, m, box[0], box[1], pts.data_ptr(), cx.stream)      # untimed
        e0.record()
        tree.QueryDevice(pts.data_ptr(), m, out.data_ptr(), cx.stream)
        e1.record()
        torch.cuda.synchronize()
        q_ms += e0.elapsed_time(e1)
        bits += out[:m].view(torch.int64).sum()           # wraps mod 2^64: an order-independent checksum of the value BITS
        done += m
    if cx.dist is not None:
        cx.dist.all_reduce(bits, op=cx.dist.ReduceOp.SUM)
    q_ms = cx.max_over_ranks(q_ms)[0]
    hbm_peak, _ = peaks()
    return {"points": total, "ms": q_ms, "points_per_s": total / (q_ms * 1e-3), "scaling": "strong",
            "tree": "C3 octree replicated on every rank; points = Philox4x32-10(seed 0x5DF0C7EE, counter = global index), sharded contiguously",
            "hbm_GBps_per_gpu": total / cx.world * 32 / (q_ms * 1e-3) / 1e9, "frac_of_hbm_peak": total / cx.world * 32 / (q_ms * 1e-3) / 1e9 / hbm_peak,
            "checksum_int64_of_value_bits": int(bits.cpu()[0])}


def query_flops_per_point(hp, tree):
    """Algorithmic FP64 flops of one Query on `tree`, averaged over uniform points of the root box: per leaf of degree p the
    three Legendre recurrences (about 3 flops per degree and axis: 9p) and the N_p-term sum sum c * Lx * Ly * Lz (4 N_p),
    weighted by the leaf's share of the volume (SURVEY.md 8d)."""
    nodes = hp.parse_block(tree.ToMemoryBlockBytes())["nodes"]
    leaf = nodes["child"] == NOCHILD
    ext = (nodes["mx"][leaf] - nodes["mn"][leaf]).astype(np.float64)
    vol = ext.prod(1)
    deg = nodes["deg"][leaf].astype(np.int64)
    ncoef = np.asarray(hp.COEFF_COUNT)[deg]
    return float(((9 * deg + 4 * ncoef) * vol).sum() / vol.sum())


def bench_query(cx, tree, box, fp64_peak, label):
    """2^24-point launches (inputs larger than L2), device-resident Philox points: the HBM roofline of queryKernel, plus the
    host-buffer e2e through hpsdf_query."""
    hp, torch = cx.hp, cx.torch
    n_q = QUERY_POINTS
    pts = torch.empty((n_q, 3), device="cuda", dtype=torch.float64)
    out = torch.empty(n_q, device="cuda", dtype=torch.float64)
    hp.uniform_points_device(SEED, cx.rank * n_q, n_q, box[0], box[1], pts.data_ptr(), cx.stream)
    for _ in range(3):
        tree.QueryDevice(pts.data_ptr(), n_q, out.data_ptr(), cx.stream)
    cx.barrier()
    q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    q0.record()
    for _ in range(reps):
        tree.QueryDevice(pts.data_ptr(), n_q, out.data_ptr(), cx.stream)
    q1.record()
    cx.barrier()
    q_ms = cx.max_over_ranks(q0.elapsed_time(q1) / reps)[0]
    import ctypes
    n_qe = 1 << 22
    hpts = torch.empty((n_qe, 3), dtype=torch.float64).pin_memory()
    hpts.copy_(pts[:n_qe].cpu())
    hout = torch.empty(n_qe, dtype=torch.float64).pin_memory()
    for i in range(4):
        if i == 1:
            cx.barrier()
            tq0 = time.perf_counter()
        hp._check(hp.lib().hpsdf_query(tree._h, ctypes.c_void_p(hpts.data_ptr()), n_qe, ctypes.c_void_p(hout.data_ptr())))
    qe_s = cx.max_over_ranks((time.perf_counter() - tq0) / 3)[0]
    hbm_peak, peak_src = peaks()
    q_flops = query_flops_per_point(hp, tree)
    gbs = n_q * 32 / (q_ms * 1e-3) / 1e9
    return {"metric": "query_points_per_s", "tree": label, "value": cx.world * n_q / (q_ms * 1e-3), "unit": "points/s", "points_per_gpu": n_q,
            "ms": q_ms, "scaling": "weak",
            "e2e": {"value": cx.world * n_qe / qe_s, "unit": "points/s", "h2d_bytes_per_step": n_qe * 24, "d2h_bytes_per_step": n_qe * 8},
            "roofline": {"kernel": "queryKernel", "bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                         "algorithmic_bytes_per_launch": n_q * 32,
                         # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this launch shape (2^24 points,
                         # C2 tree): profiles/r2_query_kernel.md. Not re-measured in this run.
                         "traffic": NCU_QUERY_TRAFFIC_BYTES if n_q == (1 << 24) else None,
                         "traffic_source": "profiles/r2_query_kernel.md (405.7 MB read + 119.5 MB written per 2^24-point launch)", "peak_source": peak_src,
                         "fp64": {"algorithmic_flops_per_point": q_flops, "achieved": q_flops * n_q / (q_ms * 1e-3) / 1e12,
                                  "peak": fp64_peak, "unit": "TFLOP/s", "frac": q_flops * n_q / (q_ms * 1e-3) / 1e12 / fp64_peak}}}


def bench_c2(cx, args, fp64_peak, with_cpu):
    """configs[1]: closed-form CSG, fit kernels specialised to the program at run time (NVRTC). Reports the cold start."""
    hp, torch = cx.hp, cx.torch
    cfg, prog = product_case(hp, "c2_csg")
    opts = cx.opts(jit=1)
    tree = hp.Octree()
    jit_note = "fit kernels specialised to the SDF program at run time (NVRTC)"
    t0 = time.perf_counter()
    try:
        tree.Create(cfg, prog, opts)
    except hp.HpsdfError as e:
        jit_note = "unavailable (%s): interpreted fit kernels" % e
        opts.jit = 2
        tree.Create(cfg, prog, opts)
    cold_s = time.perf_counter() - t0
    ms, agg = cx.timed_creates(tree, cfg, prog, opts, args.steps, args.warmup)
    st = tree.stats()
    fits = useful_fits(st)
    e2e = []
    for i in range(max(3, min(args.steps, 10))):
        t0 = time.perf_counter()
        t2 = hp.Octree()
        t2.Create(cfg, prog, opts)
        blk = t2.ToMemoryBlock()
        torch.cuda.synchronize()
        e2e.append(time.perf_counter() - t0)
        blk_bytes = blk.size
        blk.free()
        t2.Clear()
    e2e_ms = cx.max_over_ranks(1e3 * float(np.mean(e2e[1:])))[0]
    fit_tflops = agg["algorithmic_flops"] / max(agg["fit_kernel_ms"] * 1e-3, 1e-12) / 1e12
    res = {"workload": "c2_csg", "ms_per_step": ms, "fits_per_s": fits / (ms * 1e-3), "nodes_fitted_per_step": fits,
           "fits_evaluated_per_step": st["fits_evaluated"], "rounds": st["rounds"], "n_nodes": st["n_nodes"], "n_coeffs": st["n_coeffs"],
           "jit": jit_note, "cold_start_s": cold_s, "jit_compile_s": max(cold_s - ms * 1e-3, 0.0),
           "e2e": {"value": fits / (e2e_ms * 1e-3), "unit": "fits/s", "ms_per_step": e2e_ms,
                   "h2d_bytes_per_step": int(80 + 80 * len(CASES["c2_csg"]["prog"]) + 32 * st["jobs_evaluated"]),
                   "d2h_bytes_per_step": int(blk_bytes + 16 * st["fits_evaluated"])},
           "host_ms_per_step": {k: agg[k] / args.steps for k in ("host_replay_ms", "host_select_ms", "host_tasks_ms", "device_wait_ms", "pack_ms", "finalize_ms", "fit_kernel_ms")},
           "gpu_busy_frac": agg["fit_kernel_ms"] / args.steps / ms,
           "roofline": {"kernel": "fitKernel<D> specialised to the program (all fit launches of the timed builds)", "bound": "fp64",
                        "achieved": fit_tflops, "peak": fp64_peak, "unit": "TFLOP/s", "frac": fit_tflops / fp64_peak,
                        # FP64 on the CUDA cores (tcgen05 has no FP64 kind): neither of the contract's "hbm" / "tensor"; DRAM traffic of
                        # these kernels is 32 B read per fit (ncu: 8.4 MB for 262 144 fits, profiles/r2_fit_kernel_jit.md), so no HBM figure
                        "traffic": None, "peak_source": "DFMA rate measured in this run (dfmaPeakKernel); MEASURED_PEAKS.json holds no FP64 figure",
                        "whole_step_frac": agg["algorithmic_flops"] / args.steps / (ms * 1e-3) / 1e12 / fp64_peak}}
    frontier = {}
    if cx.rank == 0:
        hp.set_jit(opts.jit == 1)
        for p in (2, 3, 4):
            fb = hp.bench_frontier(cfg, prog, 5, p, repeats=3, device=cx.local, stream=cx.stream)
            tf = fb["algorithmic_flops"] / (fb["ms_per_launch"] * 1e-3) / 1e12
            frontier["p%d" % p] = {"ms": fb["ms_per_launch"], "jobs": fb["jobs"], "fits_per_s": fb["fits"] / (fb["ms_per_launch"] * 1e-3),
                                   "sdf_evals_per_s": fb["sdf_evals"] / (fb["ms_per_launch"] * 1e-3), "algorithmic_tflops": tf,
                                   "frac_of_fp64_peak": tf / fp64_peak}
        hp.set_jit(False)
    res["roofline_frontier"] = frontier
    if with_cpu:
        dt, kind, ctree = cpu_reference_build(os.cpu_count() or 1, "c2_csg")
        cq = np.random.default_rng(1).uniform(-0.25, 0.5, (2_000_000, 3))
        t0 = time.perf_counter()
        ctree.query(cq, os.cpu_count() or 1)
        res["cpu_baseline"] = {"value": fits / dt, "unit": "fits/s", "cores": os.cpu_count() or 1, "kind": kind,
                               "sample": "one full stock Octree::Create of c2_csg (%.2f s)" % dt,
                               "query_points_per_s": len(cq) / (time.perf_counter() - t0)}
    return res, tree


def bench_c1(cx, args, with_cpu):
    """configs[0]: README sphere, threshold 1e-6, exponential nearness 3.0, continuity strength 8."""
    hp = cx.hp
    cfg, prog = product_case(hp, "c1_readme")
    tree = hp.Octree()
    ms, agg = cx.timed_creates(tree, cfg, prog, cx.opts(jit=1), args.steps, args.warmup)
    st = tree.stats()
    fits = useful_fits(st)
    res = {"workload": "c1_readme", "ms_per_step": ms, "fits_per_s": fits / (ms * 1e-3), "nodes_fitted_per_step": fits,
           "continuity_ms": agg["continuity_ms"] / args.steps, "continuity_cg_ms": agg["continuity_cg_ms"] / args.steps,
           "continuity_assembly_ms": agg["continuity_assembly_ms"] / args.steps, "continuity_enum_ms": agg["continuity_enum_ms"] / args.steps,
           "cg_iterations": st["cg_iterations"], "n_nodes": st["n_nodes"], "n_coeffs": st["n_coeffs"]}
    if with_cpu:
        dt, kind, _ = cpu_reference_build(os.cpu_count() or 1, "c1_readme")
        res["cpu_baseline"] = {"value": fits / dt, "unit": "fits/s", "cores": os.cpu_count() or 1, "kind": kind,
                               "sample": "one full stock Octree::Create of c1_readme incl. its continuity post-process (%.2f s)" % dt, "ms": 1e3 * dt}
    return res


def bench_c4(cx, with_cpu):
    hp = cx.hp
    verts, tris, box, cfg = mesh_case(cx, MESH_C4_UV, C4)
    t0 = time.perf_counter()
    mesh = hp.Mesh(verts, tris, device=cx.local)
    setup_s = time.perf_counter() - t0
    prog = hp.SdfProgram([("mesh", [], mesh)])
    tree = hp.Octree()
    ms, agg = cx.timed_creates(tree, cfg, prog, cx.opts(max_degree=C4["max_degree"]), 1, 1)
    st = tree.stats()
    fits = useful_fits(st)
    res = {"workload": "c4_ramesses_standin", "triangles": int(len(tris)), "threshold": C4["threshold"], "max_degree": C4["max_degree"],
           "ms_per_step": ms, "fits_per_s": fits / (ms * 1e-3), "nodes_fitted_per_step": fits, "fits_evaluated": st["fits_evaluated"],
           "mesh_sdf_evals": st["sdf_evals"], "mesh_sdf_evals_per_s": st["sdf_evals"] / (ms * 1e-3),
           "fit_and_sample_kernel_ms": st["fit_kernel_ms"], "rounds": st["rounds"], "n_nodes": st["n_nodes"], "n_coeffs": st["n_coeffs"],
           "mesh_setup_s": setup_s, "e2e_ms": 1e3 * setup_s + ms, "scaling": "strong",
           "step_breakdown_ms": {k: agg[k] for k in ("fit_kernel_ms", "continuity_ms", "continuity_cg_ms", "continuity_assembly_ms",
                                                      "continuity_enum_ms", "device_wait_ms", "pack_ms", "finalize_ms") if k in agg}}
    if with_cpu:
        try:
            res["cpu_baseline"] = cpu_fit_sample(hp, tree, verts, tris, box, C4, budget_s=12.0)
        except Exception as e:
            res["cpu_baseline"] = {"unavailable": repr(e)}
    return res


def cpu_reference_build(threads, name):
    """The reference's own Octree::Create (unmodified sources, oracle/_ref, -O3 + OpenMP build) on the host cores; falls
    back to the C port when oracle/_ref was not built. Returns (seconds, kind, tree)."""
    from oracle import hpref
    c = CASES[name]
    cfg = hpref.make_config(threads=threads, **c["cfg"])
    prog = hpref.make_program(c["prog"])
    if hpref.available(fast=True):
        t0 = time.perf_counter()
        t = hpref.RefTree.build(cfg, prog, mode=0, threads=threads, fast=True)
        return time.perf_counter() - t0, "reference", t
    from oracle import hporacle
    t0 = time.perf_counter()
    t = hporacle.OracleTree.build(cfg, prog, threads=threads)
    return time.perf_counter() - t0, "port", t


def run_reference_arm(args):
    """The stock reference on the host cores: Mesh::CreateHalfEdges + BVH::Create once, then its own Octree::Create of the
    headline workload with F = Mesh::SignedDistanceAtPt (BVH overload), threadCount = all cores. One Create takes about a
    minute, so the run is bounded to 240 s: as many full Creates as fit (at least one), no warm-up step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import hpref, hporacle
    from meshgen import bumpy_torus, mesh_root
    threads = os.cpu_count() or 1
    cfgd = headline_config()
    verts, tris = bumpy_torus(*MESH_UV)
    mn, mx = mesh_root(verts)
    fast = hpref.available(fast=True)
    kind = "reference" if fast else "port"
    t0 = time.perf_counter()
    if fast:
        rm = hpref.RefMesh.create(verts, tris, True, fast=True)
        handle = rm.h
    else:
        rm = hporacle.OracleMesh(verts, tris)
        handle = rm.h
    setup_s = time.perf_counter() - t0
    cfg = hpref.make_config(threshold=C3["threshold"], nearness=0, strength=0.0, continuity=C3["continuity"], cstrength=C3["cstrength"],
                            threads=threads, root_min=mn, root_max=mx)
    prog = hpref.make_program([("mesh", [], handle)])
    times, budget_s, t_start = [], 240.0, time.perf_counter()
    tree = None
    for i in range(max(args.steps, 1)):
        t0 = time.perf_counter()
        if fast:
            tree = hpref.RefTree.build(cfg, prog, mode=0, threads=threads, fast=True)
        else:
            tree = hporacle.OracleTree.build(cfg, prog, threads=threads)
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start + times[-1] > budget_s:
            break
    ms = 1e3 * float(np.mean(times))
    n_nodes = int(hpref.parse_block(tree.block())["n_nodes"])
    fits = cfgd["nodes_fitted_per_step"]
    if not fits:
        fits = 4096 + 9 * ((n_nodes - 4681) // 8)          # lower bound from the tree alone (H jobs only) when the fixture is absent
    value = fits / (ms * 1e-3)
    npts = 2_000_000
    pts = np.random.default_rng(SEED).uniform(mn, mx, (npts, 3))
    t0 = time.perf_counter()
    tree.query(pts, threads)
    qv = npts / (time.perf_counter() - t0)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "fits/s", "n_gpus": 0, "steps": len(times),
        "warmup": 0, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": cfgd,
        "cpu_baseline": {"value": value, "unit": "fits/s", "cores": threads, "kind": kind,
                         "sample": "%d full stock Octree::Create of %s (%.1f s each; literal asynchronous schedule: built %d nodes), "
                                   "mesh + BVH set-up %.1f s outside the timed region" % (len(times), WORKLOAD, ms * 1e-3, n_nodes, setup_s)},
        "e2e": {"value": fits / (ms * 1e-3 + setup_s), "unit": "fits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "what": "CreateHalfEdges + BVH::Create + Octree::Create per step"},
        "query": {"metric": "query_points_per_s", "value": qv, "unit": "points/s", "points": npts, "threads": threads},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--only", default="", help="comma list of legs to run besides the headline: c1,c2,c4,c5,query (default: all)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the headline tree of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
        return
    args.warmup = max(args.warmup, 3)
    legs = set(args.only.split(",")) if args.only else {"c1", "c2", "c4", "c5", "query"}

    cx = Ctx()
    hp = cx.hp
    with_cpu = cx.world == 1 and cx.rank == 0 and not args.no_cpu_baseline
    fp64_peak = hp.measure_fp64_peak(cx.local, cx.stream)
    clk = []
    c3, tree3, mesh3, verts3, tris3, box3, cfg3 = bench_c3(cx, args, clk)
    if args.dump_outputs and cx.rank == 0:
        dump_outputs(hp, tree3, args.dump_outputs)
    st = c3["stats"]
    cpu3 = None
    if with_cpu:
        try:
            cpu3 = cpu_fit_sample(hp, tree3, verts3, tris3, box3, C3, budget_s=15.0)
        except Exception as e:
            cpu3 = {"unavailable": repr(e)}
    q3 = bench_query(cx, tree3, box3, fp64_peak, "C3 octree") if "query" in legs else None
    c5 = bench_c5(cx, tree3, box3) if "c5" in legs else None
    del tree3, mesh3
    c2, tree2 = bench_c2(cx, args, fp64_peak, with_cpu) if "c2" in legs else (None, None)
    q2 = bench_query(cx, tree2, ((-0.25,) * 3, (0.5,) * 3), fp64_peak, "C2 octree") if ("query" in legs and tree2 is not None) else None
    c1 = bench_c1(cx, args, with_cpu) if "c1" in legs else None
    c4 = bench_c4(cx, with_cpu) if "c4" in legs else None

    if cx.rank == 0:
        cfgd = headline_config()
        known = cfgd["nodes_fitted_per_step"]
        agg = c3["agg"]
        evals_per_s = agg["sdf_evals"] / cx.world / max(agg["fit_kernel_ms"] * 1e-3, 1e-12)
        line = {
            "metric": METRIC, "value": c3["fits"] / (c3["ms_per_step"] * 1e-3), "unit": "fits/s", "n_gpus": cx.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": c3["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": cfgd,
            "workload_check": {"nodes_fitted_this_run": c3["fits"], "matches_fixture": (known == c3["fits"]) if known else None,
                               "n_nodes": st["n_nodes"], "n_coeffs": st["n_coeffs"], "rounds": st["rounds"], "fits_evaluated": st["fits_evaluated"]},
            "clocks": clk[0],
            "e2e": c3["e2e"],
            "gpu_launches": int(agg["kernel_launches"]),
            "cold_start": {"mesh_setup_s": c3["mesh_setup_s"], "jit_compile_s": c2["jit_compile_s"] if c2 else None,
                           "note": "once per mesh / per (SDF program, degree); outside `value`, inside `e2e` (mesh set-up)"},
            "step_breakdown_ms": {k: agg[k] / args.steps for k in ("fit_kernel_ms", "continuity_ms", "continuity_cg_ms", "continuity_assembly_ms",
                                                                   "continuity_enum_ms", "host_replay_ms", "host_select_ms", "host_tasks_ms",
                                                                   "device_wait_ms", "pack_ms", "finalize_ms")},
            "dominant_kernel": {"kernel": "meshSampleKernel", "mesh_sdf_evals_per_step": agg["sdf_evals"] / args.steps,
                                "mesh_sdf_evals_per_s_per_gpu_kernel_time": evals_per_s,
                                "note": "closest-triangle BVH traversal: bound by dependent L2 round trips and divergence, neither HBM nor FP64 "
                                        "(profiles/r2_mesh_sample_kernel.md); SURVEY.md 8d: report evaluations/s"},
            "roofline": (c2 or {}).get("roofline"),
            "roofline_note": "north_star: FP64 peak for fitting (fit kernels measured on configs[1], closed-form SDF evaluated in registers; peak = DFMA "
                             "rate measured in this run, MEASURED_PEAKS.json holds no FP64 figure), HBM for Query (`query.roofline`)",
            "query": q3, "query_c2_tree": q2, "c5_query_1e9": c5, "c1_readme": c1, "c2_csg": c2, "c4_ramesses_standin": c4,
        }
        if "multi_gpu_parity" in c3:
            line["multi_gpu_parity"] = c3["multi_gpu_parity"]
        if cpu3 is not None:
            line["cpu_baseline"] = cpu3
        print(json.dumps(line))
    if cx.comm is not None:
        cx.comm.close()
    if cx.dist is not None:
        cx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
