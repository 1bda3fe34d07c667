"""Isosurface extraction on the C3 and C2 trees (GPU box): python tools/isosurface_sparse_bench.py [--sizes N ...] [--reps R]
[--label L] [--out FILE.json]

C3 is built as tools/isosurface_bench.py builds it, C2 is the c2_csg case. Both entry points pick the dense or the sparse
pipeline by grid-point count (DESIGN §15). To measure one pipeline alone at every size, load a library built with
HPSDF_ISO_SPARSE_MIN_POINTS=0 (always sparse) or =0xFFFFFFFFFFFFFFFFull (dense up to 1024 cells per axis) through HPSDF_LIB, and
alternate such runs. Per size: one warm-up call, then R calls (host clock around the blocking call from Python), with the
phase times, active blocks per culling level and peak scratch from the library's HPSDF_ISO_TIMES lines. Prints one JSON
object, with the card's name and power limit."""
import argparse
import importlib
import json
import os
import re
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402

hp = importlib.import_module("hp-adaptive-signed-distance-field-octree_b200")
from common import product_cfg  # noqa: E402
from isosurface_bench import card  # noqa: E402
from meshgen import bumpy_torus, mesh_root  # noqa: E402

DENSE = re.compile(r"grid ([\d.]+) ms, count\+scan ([\d.]+) ms, emit ([\d.]+) ms, copy ([\d.]+) ms")
SPARSE = re.compile(r"culling ([\d.]+) ms \(uncertified / blocks by edge ([^)]*)\), block pass ([\d.]+) ms, scans ([\d.]+) ms, "
                    r"emit ([\d.]+) ms, copy ([\d.]+) ms; (\d+) active blocks, \d+ \+ \d+ rows, peak scratch (\d+) bytes")


class Captured:
    """stderr of the library into a temporary file while the HPSDF_ISO_TIMES lines are wanted."""
    def __enter__(self):
        os.environ["HPSDF_ISO_TIMES"] = "1"
        self.saved, self.log = os.dup(2), tempfile.TemporaryFile(mode="w+")
        os.dup2(self.log.fileno(), 2)
        return self

    def __exit__(self, *exc):
        os.dup2(self.saved, 2)
        os.close(self.saved)
        del os.environ["HPSDF_ISO_TIMES"]
        self.log.seek(0)
        self.text = self.log.read()
        self.log.close()


def timed(fn, n):
    t0 = time.perf_counter()
    out = fn(n)
    return (time.perf_counter() - t0) * 1e3, out


def sparse_row(m):
    levels = [dict(zip(("cells", "uncertified", "blocks"), (int(a), int(b), int(c)))) for a, b, c in
              re.findall(r"(\d+): (\d+) / (\d+)", m.group(2))]
    for lv in levels:
        lv["active_fraction"] = lv["uncertified"] / lv["blocks"]
    return {"culling": float(m.group(1)), "block_pass": float(m.group(3)), "scans": float(m.group(4)), "emit": float(m.group(5)),
            "copy": float(m.group(6)), "active_blocks": int(m.group(7)), "peak_scratch_bytes": int(m.group(8)), "levels": levels}


def run(tree, n, reps):
    with Captured() as cap:
        walls = []
        for _ in range(reps + 1):
            ms, out = timed(tree.ExtractIsosurfaceSparse, n)
            walls.append(ms)
    d = [[float(x) for x in m.groups()] for m in DENSE.finditer(cap.text)][1:]
    s = [sparse_row(m) for m in SPARSE.finditer(cap.text)][1:]
    row = {"resolution": n, "vertices": len(out[0]), "triangles": len(out[1]), "pipeline": "sparse" if s else "dense",
           "ms_per_call": float(np.mean(walls[1:])), "ms_median": float(np.median(walls[1:])), "ms_calls": walls[1:]}
    if s:
        row["phase_ms"] = {k: float(np.mean([r[k] for r in s])) for k in ("culling", "block_pass", "scans", "emit", "copy")}
        row["sparse_detail"] = s[-1]
    else:
        row["phase_ms"] = dict(zip(("grid", "count_scan", "emit", "copy"), np.mean(d, 0).tolist()))
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--sizes", type=int, nargs="+", default=[256, 320, 384, 448, 512, 1024, 2048, 4096])
    ap.add_argument("--label", default="dispatch")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    verts, tris = bumpy_torus(1000, 435)
    lo, hi = mesh_root(verts)
    c3 = hp.Octree()
    c3.Create(hp.Config(target_error_threshold=1e-6, nearness_type=0, nearness_strength=0.0, continuity_enforce=1, continuity_strength=8.0,
                        thread_count=os.cpu_count() or 1, root_min=lo, root_max=hi), hp.SdfProgram([("mesh", [], hp.Mesh(verts, tris))]),
              hp.BuildOpts(max_degree=11))
    c2 = hp.Octree()
    c2.Create(*product_cfg(hp, "c2_csg"))
    res = {"card": card(), "label": a.label, "lib": os.environ.get("HPSDF_LIB", "default build"), "reps": a.reps, "trees": {}}
    for name, tree, desc in (("C3", c3, "bumpy torus U=1000 V=435 (870 000 triangles), threshold 1e-6, continuity 8, max degree 11"),
                             ("C2", c2, "tests/cases.py c2_csg")):
        t0 = time.perf_counter()
        tree.QueryBounds(np.zeros((1, 3)), np.zeros((1, 3)))                  # the bounds table, built once per tree
        entry = {"description": desc, "nodes": tree.stats()["n_nodes"], "bounds_table_ms": (time.perf_counter() - t0) * 1e3, "runs": []}
        res["trees"][name] = entry
        for n in a.sizes:
            entry["runs"].append(run(tree, n, a.reps))
            print(a.label, name, json.dumps({k: v for k, v in entry["runs"][-1].items() if k != "sparse_detail"}), flush=True)
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
