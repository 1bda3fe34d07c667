"""hpsdf_query_device against hpsdf_query_derivatives_device (ORDER 1: value + gradient, ORDER 2: + Hessian) on the C3 tree
(870 k-triangle bumpy torus, threshold 1e-6, as tools/raycast_bench.py builds it), and Octree.QueryTorch forward + backward
against the bare launches (GPU box):
python tools/derivatives_bench.py [--window S] [--out FILE.json]

Point sets, 2^26 points each (1.5 GB of input, far beyond the 126 MB L2): Philox points uniform in the root
(hpsdf_uniform_points_device), and a coherent grid of 512 x 512 x 256 points over the root in x-rows (x fastest, as the
isosurface grid pass visits them). Each launch is warmed up, then repeated for about --window seconds between CUDA events.
Algorithmic bytes per point: 24 in, plus 8 (Query), 32 (ORDER 1) or 80 (ORDER 2) out. Prints one JSON line with the card's
name, power limit and max SM clock read in the same call."""
import argparse
import importlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

hp = importlib.import_module("hp-adaptive-signed-distance-field-octree_b200")
from meshgen import bumpy_torus, mesh_root  # noqa: E402


def card():
    return subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()


def timed(run, window):
    """ms per call of run() over about `window` seconds, after a warm-up."""
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
    return e0.elapsed_time(e1) / reps, reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--window", type=float, default=1.0)
    ap.add_argument("--log2n", type=int, default=26)
    ap.add_argument("--torch-log2n", type=int, default=24)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    verts, tris = bumpy_torus(1000, 435)
    lo, hi = mesh_root(verts)
    tree = hp.Octree()
    tree.Create(hp.Config(target_error_threshold=1e-6, nearness_type=0, nearness_strength=0.0, continuity_enforce=1, continuity_strength=8.0,
                          thread_count=os.cpu_count() or 1, root_min=lo, root_max=hi),
                hp.SdfProgram([("mesh", [], hp.Mesh(verts, tris))]), hp.BuildOpts(max_degree=11))
    lo64, hi64 = np.asarray(lo, np.float64), np.asarray(hi, np.float64)
    n = 1 << a.log2n
    s = torch.cuda.current_stream().cuda_stream
    sets = {}
    x = torch.empty((n, 3), dtype=torch.float64, device="cuda")
    hp.uniform_points_device(2024, 0, n, lo64, hi64, x.data_ptr(), s)
    sets["philox_uniform"] = x
    nx, ny = 512, 512
    nz = n // (nx * ny)
    axes = [torch.linspace(float(lo64[i]), float(hi64[i]), m, dtype=torch.float64, device="cuda") for i, m in enumerate((nx, ny, nz))]
    Z, Y, X = torch.meshgrid(axes[2], axes[1], axes[0], indexing="ij")
    sets["grid_x_rows"] = torch.stack([X.reshape(-1), Y.reshape(-1), Z.reshape(-1)], 1).contiguous()
    del X, Y, Z
    v = torch.empty(n, dtype=torch.float64, device="cuda")
    g = torch.empty((n, 3), dtype=torch.float64, device="cuda")
    h = torch.empty((n, 6), dtype=torch.float64, device="cuda")
    res = {"card": card(), "lib": os.path.relpath(hp.LIB_PATH, ROOT), "window_s": a.window, "points": n,
           "tree": "C3: bumpy torus U=1000 V=435 (870 000 triangles), threshold 1e-6, continuity 8, max degree 11",
           "nodes": int(tree.stats()["n_nodes"]), "runs": {}}
    for name, pts in sets.items():
        runs = {
            "query": (lambda: tree.QueryDevice(pts.data_ptr(), n, v.data_ptr(), s), 32),
            "order1": (lambda: tree.QueryDerivativesDevice(pts.data_ptr(), n, v.data_ptr(), g.data_ptr(), None, s), 56),
            "order2": (lambda: tree.QueryDerivativesDevice(pts.data_ptr(), n, v.data_ptr(), g.data_ptr(), h.data_ptr(), s), 104),
        }
        row = {}
        for k, (run, nbytes) in runs.items():
            ms, reps = timed(run, a.window)
            row[k] = {"ms": ms, "launches": reps, "points_per_s": n / (ms * 1e-3), "algorithmic_GB_per_s": n * nbytes / (ms * 1e-3) / 1e9}
        for k in ("order1", "order2"):
            row[k]["time_vs_query"] = row[k]["ms"] / row["query"]["ms"]
        res["runs"][name] = row
    # QueryTorch forward + backward over 2^torch_log2n points against the bare ORDER-1 launch on the same points
    m = 1 << a.torch_log2n
    xt = sets["philox_uniform"][:m].clone()
    ones = torch.ones(m, dtype=torch.float64, device="cuda")

    def fwd_bwd():
        xr = xt.detach().requires_grad_(True)
        tree.QueryTorch(xr).backward(ones)

    ms_t, reps_t = timed(fwd_bwd, a.window)
    ms_1, _ = timed(lambda: tree.QueryDerivativesDevice(xt.data_ptr(), m, v.data_ptr(), g.data_ptr(), None, s), a.window)
    ms_0, _ = timed(lambda: tree.QueryDevice(xt.data_ptr(), m, v.data_ptr(), s), a.window)
    res["torch"] = {"points": m, "forward_backward_ms": ms_t, "calls": reps_t, "order1_launch_ms": ms_1, "query_launch_ms": ms_0,
                    "forward_backward_vs_order1": ms_t / ms_1}
    res["card_after"] = card()
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
