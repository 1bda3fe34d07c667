"""hpsdf_extract_isosurface on the C3 tree (870 k-triangle bumpy torus, threshold 1e-6, as bench.py builds it) at 256^3, 512^3
and 1024^3 cells (GPU box): python tools/isosurface_bench.py [--reps R] [--out FILE.json]

Per resolution: one warm-up call, then R timed calls (host clock around the blocking call) with the device time of each
phase (grid, count + scans, emit, copy) from the library's CUDA events (HPSDF_ISO_TIMES), and hpsdf_query_device on as
many uniform Philox points in the root box as the grid has points (CUDA events) for comparison. Grid points are
coherent, random query points are not. Prints one JSON object, with the card's name and power limit."""
import argparse
import importlib
import json
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

hp = importlib.import_module("hp-adaptive-signed-distance-field-octree_b200")
from meshgen import bumpy_torus, mesh_root  # noqa: E402

PHASES = re.compile(r"grid ([\d.]+) ms, count\+scan ([\d.]+) ms, emit ([\d.]+) ms, copy ([\d.]+) ms")


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    return out


def extract_timed(tree, n, reps):
    """(wall ms per call, mean phase ms [grid, count+scan, emit, copy], vertices, triangles)."""
    os.environ["HPSDF_ISO_TIMES"] = "1"
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as log:
        os.dup2(log.fileno(), 2)
        try:
            v, t = tree.ExtractIsosurface(n)                       # warm-up
            wall = []
            for _ in range(reps):
                t0 = time.perf_counter()
                v, t = tree.ExtractIsosurface(n)
                wall.append((time.perf_counter() - t0) * 1e3)
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["HPSDF_ISO_TIMES"]
        log.seek(0)
        rows = [[float(x) for x in m.groups()] for m in PHASES.finditer(log.read())][1:]
    return float(np.mean(wall)), np.mean(rows, 0).tolist(), len(v), len(t)


def query_timed(tree, n_pts, lo, hi, reps):
    pts = torch.empty((n_pts, 3), device="cuda", dtype=torch.float64)
    out = torch.empty(n_pts, device="cuda", dtype=torch.float64)
    s = torch.cuda.current_stream().cuda_stream
    hp.uniform_points_device(0x5DF0C7EE, 0, n_pts, lo, hi, pts.data_ptr(), s)
    tree.QueryDevice(pts.data_ptr(), n_pts, out.data_ptr(), s)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        tree.QueryDevice(pts.data_ptr(), n_pts, out.data_ptr(), s)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    del pts, out
    torch.cuda.empty_cache()
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--res", type=int, nargs="+", default=[256, 512, 1024])
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    verts, tris = bumpy_torus(1000, 435)
    lo, hi = mesh_root(verts)
    mesh = hp.Mesh(verts, tris)
    cfg = hp.Config(target_error_threshold=1e-6, nearness_type=0, nearness_strength=0.0, continuity_enforce=1, continuity_strength=8.0,
                    thread_count=os.cpu_count() or 1, root_min=lo, root_max=hi)
    tree = hp.Octree()
    tree.Create(cfg, hp.SdfProgram([("mesh", [], mesh)]), hp.BuildOpts(max_degree=11))
    box_lo, box_hi = np.asarray(lo, np.float32).astype(np.float64), np.asarray(hi, np.float32).astype(np.float64)
    res = {"card": card(), "tree": "C3: bumpy torus U=1000 V=435 (870 000 triangles), threshold 1e-6, continuity 8, max degree 11",
           "nodes": tree.stats()["n_nodes"], "reps": a.reps, "runs": []}
    for n in a.res:
        wall, ph, nv, nt = extract_timed(tree, n, a.reps)
        pts = (n + 1) ** 3
        q_ms = query_timed(tree, pts, box_lo, box_hi, a.reps)
        res["runs"].append({"resolution": n, "grid_points": pts, "vertices": nv, "triangles": nt, "ms_per_call": wall,
                            "phase_ms": dict(zip(("grid", "count_scan", "emit", "copy"), ph)),
                            "grid_points_per_s": pts / (ph[0] * 1e-3), "query_device_ms": q_ms,
                            "query_device_points_per_s": pts / (q_ms * 1e-3)})
        print(json.dumps(res["runs"][-1]), flush=True)
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
