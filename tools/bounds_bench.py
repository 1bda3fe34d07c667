"""hpsdf_query_bounds_device on the C3 tree (870 k-triangle bumpy torus, threshold 1e-6, as bench.py builds it) and the C2
tree (closed-form CSG) (GPU box): python tools/bounds_bench.py [--window S] [--out FILE.json]

Per tree: the one-off build of the enclosure table (the first bounds call, timed on the host around a blocking call of one
box), then boxes generated on the device from Philox points (hpsdf_uniform_points_device):
  small  2^22 boxes, edges 2^-10 .. 2^-6 of the root (log-uniform per box), positions uniform in the root;
  large  2^16 boxes, edges 1/8 .. 1 of the root;
  tiling the 32^3, 64^3 and 128^3 block tilings of the root, with the fraction certified free of the surface (f_lo > 0 or
         f_hi < 0).
Each set: one warm-up launch, then as many launches as fill about --window seconds, timed with CUDA events. Reports boxes/s,
the mean number of leaves whose extended cell meets a box (on 4096 sampled boxes, from the MemoryBlock in numpy) and the
participating (box, leaf) pairs per second that implies. Prints one JSON object, with the card's name, power limit and
max SM clock."""
import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

hp = importlib.import_module("hp-adaptive-signed-distance-field-octree_b200")
from cases import CASES  # noqa: E402
from common import product_cfg  # noqa: E402
from meshgen import bumpy_torus, mesh_root  # noqa: E402

L = 0.5 + 2.0 ** -25


def card():
    return subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()


def philox(seed, n, lo, hi):
    out = torch.empty((n, 3), dtype=torch.float64, device="cuda")
    hp.uniform_points_device(seed, 0, n, lo, hi, out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    return out


def leaf_cells(blk):
    nodes = blk["nodes"]
    leaf = nodes["deg"] != 13
    mn, mx = nodes["mn"][leaf].astype(np.float64), nodes["mx"][leaf].astype(np.float64)
    return np.where(mn == -0.5, -L, mn), np.where(mx == 0.5, L, mx)


def time_boxes(tree, lo, hi, window):
    n = lo.shape[0]
    f_lo = torch.empty(n, dtype=torch.float64, device="cuda")
    f_hi = torch.empty(n, dtype=torch.float64, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    run = lambda: tree.QueryBoundsDevice(lo.data_ptr(), hi.data_ptr(), n, f_lo.data_ptr(), f_hi.data_ptr(), stream=s)
    run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); run(); e1.record(); torch.cuda.synchronize()
    reps = max(3, int(window / max(e0.elapsed_time(e1) * 1e-3, 1e-6)))
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, reps, f_lo, f_hi


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--window", type=float, default=1.0)
    ap.add_argument("--sample", type=int, default=4096)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    trees = []
    verts, tris = bumpy_torus(1000, 435)
    lo, hi = mesh_root(verts)
    c3 = hp.Octree()
    c3.Create(hp.Config(target_error_threshold=1e-6, nearness_type=0, nearness_strength=0.0, continuity_enforce=1, continuity_strength=8.0,
                        thread_count=os.cpu_count() or 1, root_min=lo, root_max=hi),
              hp.SdfProgram([("mesh", [], hp.Mesh(verts, tris))]), hp.BuildOpts(max_degree=11))
    trees.append(("C3: bumpy torus U=1000 V=435 (870 000 triangles), threshold 1e-6, continuity 8, max degree 11", c3, (lo, hi)))
    cfg, prog = product_cfg(hp, "c2_csg")
    c2 = hp.Octree()
    c2.Create(cfg, prog)
    k = CASES["c2_csg"]["cfg"]
    trees.append(("C2: c2_csg (box + torus + capsule CSG), threshold 1e-8", c2, (k["root_min"], k["root_max"])))
    res = {"card": card(), "window_s": a.window, "runs": []}
    for label, tree, (rlo, rhi) in trees:
        rlo, rhi = np.asarray(rlo, np.float32).astype(np.float64), np.asarray(rhi, np.float32).astype(np.float64)
        ext = torch.tensor(rhi - rlo, device="cuda")
        blk = hp.parse_block(tree.ToMemoryBlockBytes())
        elo, ehi = leaf_cells(blk)
        x = np.zeros((1, 3))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        tree.QueryBounds(x, x)                 # first call: builds the table
        build_ms = (time.perf_counter() - t0) * 1e3
        t0 = time.perf_counter()
        tree.QueryBounds(x, x)
        second_ms = (time.perf_counter() - t0) * 1e3
        print(json.dumps({"tree": label, "table_build_ms_first_call": build_ms, "second_call_ms": second_ms}), flush=True)
        sets = []
        for name, n, e0, e1, seed in (("small", 1 << 22, -10, -6, 11), ("large", 1 << 16, -3, 0, 12)):
            pos = philox(seed, n, rlo, rhi)
            u = philox(seed + 100, n, [0.0] * 3, [1.0] * 3)
            edge = torch.exp2(e0 + (e1 - e0) * u[:, :1]) * ext          # log-uniform per box, the same exponent on all axes
            sets.append((name, pos - 0.5 * edge, pos + 0.5 * edge))
        for kk in (32, 64, 128):
            g = torch.arange(kk, dtype=torch.float64, device="cuda") / kk
            G = torch.stack(torch.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
            blo = torch.tensor(rlo, device="cuda") + G * ext
            sets.append(("tiling_%d^3" % kk, blo, blo + ext / kk))
        centre, inv = (rlo + rhi) / 2, 1.0 / (rhi - rlo)
        for name, lo_d, hi_d in sets:
            lo_d, hi_d = lo_d.contiguous(), hi_d.contiguous()
            ms, reps, f_lo, f_hi = time_boxes(tree, lo_d, hi_d, a.window)
            n = lo_d.shape[0]
            pick = np.random.default_rng(7).choice(n, min(a.sample, n), replace=False)
            plo = (lo_d[pick].cpu().numpy() - centre) * inv
            phi = (hi_d[pick].cpu().numpy() - centre) * inv
            leaves = np.array([((ehi >= plo[i]) & (elo <= phi[i])).all(1).sum() for i in range(len(pick))])
            boxes_s = n / (ms * 1e-3)
            row = {"tree": label, "nodes": int(blk["n_nodes"]), "leaves": int(len(elo)), "set": name, "boxes": n, "launches": reps,
                   "ms_per_launch": ms, "boxes_per_s": boxes_s, "mean_leaves_per_box": float(leaves.mean()),
                   "box_leaf_pairs_per_s": boxes_s * float(leaves.mean())}
            if name.startswith("tiling"):
                row["certified_free_fraction"] = float(((f_lo > 0) | (f_hi < 0)).double().mean())
            res["runs"].append(row)
            print(json.dumps(row), flush=True)
            del f_lo, f_hi
            torch.cuda.empty_cache()
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
