"""Times of the laser-plane calibration on the GPU.

1. l3d_fit_plane (Context.fit_plane) on n = 1e5 / 1e6 / 1e7 points (a plane with 0.3 mm noise plus 40 % uniform
   outliers, threshold 1 mm) with 1024 and 4096 hypotheses: the median of 5 calls after a warm-up call, host clock
   around the whole call (upload of the points, RANSAC, refinement, mask download; the call synchronises), and
   n * hypotheses point-hypothesis evaluations per second over the call.
2. LaserReconstructionSystem.calibrate_laser_plane on 448 captures of bench.py's config 3 (1280x720 per eye, 128
   disparities, block 9, MODE_HH, WLS, Simple extractor): median of 3 calls after a warm-up call.
Prints the card's name and power limit first, read in the same run.
Usage: python tools/plane_fit_probe.py"""
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import laser_3d_reconstruction_b200 as l3d  # noqa: E402
from laser_3d_reconstruction_b200 import _native as N, synth  # noqa: E402


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks_throttle_reasons.active"
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True)
    except OSError:
        return "nvidia-smi unavailable"
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "nvidia-smi unavailable"


def cloud(n, seed=0):
    rng = np.random.default_rng(seed)
    nrm = np.array([0.3, -0.2, 0.9]) / np.linalg.norm([0.3, -0.2, 0.9])
    a = np.cross(nrm, [1.0, 0, 0]); a /= np.linalg.norm(a)
    b = np.cross(nrm, a)
    uv = rng.uniform(-0.5, 0.5, (n, 2))
    pts = 0.7 * nrm + uv[:, :1] * a + uv[:, 1:] * b + 3e-4 * rng.standard_normal((n, 1)) * nrm
    k = int(0.4 * n)
    pts[:k] = rng.uniform(-1, 1, (k, 3)) + [0, 0, 1]
    return np.ascontiguousarray(pts)


def timed(f, reps):
    f()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        f()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def fit_times(ctx):
    for n in (100_000, 1_000_000, 10_000_000):
        pts = cloud(n)
        for hyps in (1024, 4096):
            t = timed(lambda: ctx.fit_plane(pts, 1e-3, hyps, 0), 5)
            print(json.dumps(dict(what="l3d_fit_plane", n=n, hypotheses=hyps, ms=round(1e3 * t, 3),
                                  evals_per_s=float("%.4g" % (n * hyps / t)))), flush=True)


def calibrate_time():
    W, H, D = 1280, 720, 128
    K, _ = synth.camera_model(W, H)
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "stereo_calibration.json")
        with open(path, "w") as f:
            json.dump(dict(R=np.eye(3).tolist(), T=[[-0.06], [0.0], [0.0]], camera_matrix_left=K.tolist(),
                           dist_coeffs_left=[[0.0] * 5], camera_matrix_right=K.tolist(), dist_coeffs_right=[[0.0] * 5]), f)
        cam = l3d.SingleUSBStereoCameraManager(width=2 * W, height=H, calibration_file=path, num_disparities=D, block_size=9,
                                               sgbm_mode=1, verbose=False)
        cam.initialize_offline()
    s = l3d.LaserReconstructionSystem(l3d.Config(), verbose=False)
    s.initialize(camera=cam)
    f, B = 0.8 * W, 0.06
    Z0 = f * B / (0.35 * D)
    plane = -np.array([1.0, -0.1, 0.5, -(0.05 * Z0 + 0.5 * Z0)]) / np.linalg.norm([1.0, -0.1, 0.5])
    base = [synth.plane_stripe_pair(W, H, D, plane, 0.75 + 0.5 * k / 7, seed=k) for k in range(8)]
    caps = np.stack([np.concatenate(base[i % 8][:2], axis=1) for i in range(448)])
    fit = [None]

    def run():
        fit[0] = s.calibrate_laser_plane(frames=caps)

    t = timed(run, 3)
    print(json.dumps(dict(what="calibrate_laser_plane", captures=448, geometry="1280x720 D128 block 9 MODE_HH WLS Simple",
                          ms=round(1e3 * t, 1), frames_per_s=round(448 / t, 1), points=int(len(fit[0].inlier_mask)),
                          inliers=fit[0].inliers, plane=[round(v, 6) for v in fit[0].plane],
                          true_plane=[round(v, 6) for v in plane])), flush=True)
    s.stop()


def main():
    print("card: %s" % card(), flush=True)
    ctx = N.Context(0)
    fit_times(ctx)
    ctx.close()
    calibrate_time()


if __name__ == "__main__":
    main()
