"""hpsdf_raycast_device on the C3 tree (870 k-triangle bumpy torus, threshold 1e-6, as bench.py builds it) and the C2 tree
(closed-form CSG), with pinhole-camera primary rays generated on the device at 1920x1080 and 4096^2 (GPU box):
python tools/raycast_bench.py [--window S] [--out FILE.json]

Per tree and resolution: one warm-up launch, then as many launches as fill a window of about --window seconds, timed with
CUDA events. Reports rays/s and the hit fraction; from the numpy checker (tests/raycast_ref.py) on 4096 sampled rays, the mean
number of leaves a ray visits and the mean m+1 per leaf (m = the warp's largest leaf degree, the kernel evaluates m+1 points
per leaf; the checker gives each ray's own degrees, so the mean of p+1 over a ray's leaves is reported as a lower bound of
m+1); and the point evaluations per second that implies. Prints one JSON object, with the card's name and power limit."""
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
import raycast_ref as R  # noqa: E402
from cases import CASES  # noqa: E402
from common import product_cfg  # noqa: E402
from meshgen import bumpy_torus, mesh_root  # noqa: E402


def card():
    return subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()


def pinhole_device(eye, target, w, h, fov):
    """Primary rays of a w x h pinhole camera (vertical half-angle fov), built on the device with torch."""
    eye, target = (torch.tensor(np.asarray(x, np.float64), device="cuda") for x in (eye, target))
    f = target - eye; f = f / f.norm()
    r = torch.linalg.cross(f, torch.tensor([0.0, 0.0, 1.0], dtype=torch.float64, device="cuda")); r = r / r.norm()
    u = torch.linalg.cross(r, f)
    s = float(np.tan(fov))
    xs = ((torch.arange(w, dtype=torch.float64, device="cuda") + 0.5) / w * 2 - 1) * s * w / h
    ys = ((torch.arange(h, dtype=torch.float64, device="cuda") + 0.5) / h * 2 - 1) * s
    Y, X = torch.meshgrid(ys, xs, indexing="ij")
    d = f + X.reshape(-1, 1) * r + Y.reshape(-1, 1) * u
    o = eye.expand_as(d).contiguous()
    return o, d.contiguous()


def time_rays(tree, o, d, window):
    n = o.shape[0]
    t = torch.empty(n, dtype=torch.float64, device="cuda")
    nrm = torch.empty((n, 3), dtype=torch.float64, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    run = lambda: tree.RaycastDevice(o.data_ptr(), d.data_ptr(), n, t.data_ptr(), nrm.data_ptr(), stream=s)
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
    ms = e0.elapsed_time(e1) / reps
    return ms, reps, t


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
    trees.append(("C3: bumpy torus U=1000 V=435 (870 000 triangles), threshold 1e-6, continuity 8, max degree 11", c3, (lo, hi),
                  np.array([0.35, -0.9, 0.55]), 0.3))
    cfg, prog = product_cfg(hp, "c2_csg")
    c2 = hp.Octree()
    c2.Create(cfg, prog)
    k = CASES["c2_csg"]["cfg"]
    trees.append(("C2: c2_csg (box + torus + capsule CSG), threshold 1e-8", c2, (k["root_min"], k["root_max"]),
                  np.array([0.5, -1.0, 0.6]), 0.3))
    res = {"card": card(), "window_s": a.window, "runs": []}
    for label, tree, (lo, hi), view, fov in trees:
        lo, hi = np.asarray(lo, np.float64), np.asarray(hi, np.float64)
        centre, ext = (lo + hi) / 2, (hi - lo).max()
        blk = hp.parse_block(tree.ToMemoryBlockBytes())
        llo, lhi, deg = R.tree_leaves(blk)
        for w, h in ((1920, 1080), (4096, 4096)):
            o, d = pinhole_device(centre + ext * view, centre, w, h, fov)
            ms, reps, t = time_rays(tree, o, d, a.window)
            hit = float(torch.isfinite(t).double().mean())
            pick = np.random.default_rng(7).choice(o.shape[0], a.sample, replace=False)
            ref = R.cast(o[pick].cpu().numpy(), d[pick].cpu().numpy(), tuple(lo), tuple(hi), llo, lhi, deg, tree.Query,
                         scale=float(np.linalg.norm(hi - lo)))
            leaves = float(ref["leaves"].mean())
            per_leaf = [p + 1 for ds in ref["degrees"] for p in ds]
            mp1 = float(np.mean(per_leaf)) if per_leaf else 0.0
            rays_s = o.shape[0] / (ms * 1e-3)
            row = {"tree": label, "nodes": int(blk["n_nodes"]), "resolution": [w, h], "rays": int(o.shape[0]), "launches": reps,
                   "ms_per_launch": ms, "rays_per_s": rays_s, "hit_fraction": hit,
                   "checker_sample": a.sample, "checker_hit_fraction": float(np.isfinite(ref["t"]).mean()),
                   "mean_leaves_per_ray": leaves, "mean_p_plus_1_per_leaf": mp1,
                   "implied_point_evals_per_s_lower_bound": rays_s * leaves * mp1}
            res["runs"].append(row)
            print(json.dumps(row), flush=True)
            del o, d, t
            torch.cuda.empty_cache()
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
