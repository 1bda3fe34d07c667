"""How far from orthonormal the f32 frames of decodeFrame (csrc/mesh_eval.cuh) are, and how far encodeFrame turns a frame.

The decode is restated in numpy float32: every operation of it is a correctly rounded IEEE f32 operation (rcpRnSmall
included), so the emulation has the device's bits. For N random codes of the fundamental zone (|x|, |y|, |z| <= sqrt(2) - 1,
the only codes encodeFrame produces) it prints the largest singular value of the decoded frame minus 1, in float64.
Usage: python tools/frame_sweep.py [N]   (default 5e7, about 2 minutes)"""
import sys
import time

import numpy as np

f = np.float32
N = int(float(sys.argv[1])) if len(sys.argv) > 1 else 50_000_000
lim = np.sqrt(2.0) - 1.0
rng = np.random.default_rng(0)
worst, t0, done = 0.0, time.time(), 0
while done < N:
    n = min(2_000_000, N - done)
    cx = np.clip(np.rint(rng.uniform(-lim, lim, n) * 2048) + 1024, 0, 2047)
    cy = np.clip(np.rint(rng.uniform(-lim, lim, n) * 2048) + 1024, 0, 2047)
    cz = np.clip(np.rint(rng.uniform(-lim, lim, n) * 1024) + 512, 0, 1023)
    x, y, z = ((cx - 1024) / 2048).astype(f), ((cy - 1024) / 2048).astype(f), ((cz - 512) / 1024).astype(f)
    xx, yy, zz, xy, xz, yz = x * x, y * y, z * z, x * y, x * z, y * z
    px, mx = f(1) + xx, f(1) - xx
    s = f(1) / (px + (yy + zz))
    t = f(2) * s
    F = np.empty((n, 3, 3), np.float64)
    F[:, 0, 0] = (px - (yy + zz)) * s; F[:, 0, 1] = (xy - z) * t; F[:, 0, 2] = (xz + y) * t
    F[:, 1, 0] = (xy + z) * t; F[:, 1, 1] = (mx + (yy - zz)) * s; F[:, 1, 2] = (yz - x) * t
    F[:, 2, 0] = (xz - y) * t; F[:, 2, 1] = (yz + x) * t; F[:, 2, 2] = (mx - (yy - zz)) * s
    lam = np.linalg.eigvalsh(F @ F.transpose(0, 2, 1))[:, -1]
    worst = max(worst, float((np.sqrt(lam) - 1.0).max()))
    done += n
print("codes %d: max singular value - 1 = %.3e (%.2f * 2^-24); %.0f s" % (done, worst, worst / 2.0 ** -24, time.time() - t0))
