"""Wide disparity ranges (numDisparities in (256, 512]) on the direction-split path: steady-state frames/s of the frame
pipeline, single-frame compute_depth latency, and the per-launch times of the aggregation kernels, every kernel timed
alone (pipeline timing mode).  Prints the card, its power limit and SM clock first.
Usage: L3D_PROBE_GEOM=W,H,D,BS L3D_PROBE_MODES=1,2 python tools/wide_probe.py [lanes] [frames]
(default 1920,1080,384,11, modes MODE_HH and SGBM_3WAY, 4 lanes, 16 frames)"""
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from laser_3d_reconstruction_b200 import _native as N, pipeline, synth  # noqa: E402

W, H, D, BS = (int(v) for v in os.environ.get("L3D_PROBE_GEOM", "1920,1080,384,11").split(","))
MODES = [int(m) for m in os.environ.get("L3D_PROBE_MODES", "1,2").split(",")]
lanes = int(sys.argv[1]) if len(sys.argv) > 1 else 4
nfr = int(sys.argv[2]) if len(sys.argv) > 2 else 16
GROUPS = ["sgbm_cost", "sgbm_scan_k0", "sgbm_scan_k2", "sgbm_scan_k3", "sgbm_scan_k4", "sgbm_scan_k5", "sgbm_scan_k6",
          "sgbm_scan_k7", "sgbm_wta", "wls"]


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks_throttle_reasons.active"
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True)
    except OSError:
        return "nvidia-smi unavailable"
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "nvidia-smi unavailable"


def main():
    print("card: %s" % card(), flush=True)
    print("geometry %dx%d D %d block %d, %d lanes, %d frames per run" % (W, H, D, BS, lanes, nfr), flush=True)
    K, Q = synth.camera_model(W, H)
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    base = [synth.stereo_pair(W, H, D, s) for s in range(4)]  # the matcher's work does not depend on the content
    L = np.stack([base[i % 4][0] for i in range(nfr)])
    R = np.stack([base[i % 4][1] for i in range(nfr)])
    ctx = N.Context(0)
    for mode in MODES:
        cfg = pipeline.make_pipeline_config(W, H, D, BS, mode, Q, K, lanes=lanes, max_points=20000, extractor=N.STEGER_IMPROVED)
        fp = pipeline.FramePipeline(cfg, maps=maps, ctx=ctx)
        try:
            dL, dR = fp.upload(L), fp.upload(R)
            for _ in range(3):
                fp.run_dev(dL, dR, nfr)
            ms = []
            for _ in range(5):
                fp.run_dev(dL, dR, nfr)
                ms.append(fp.last_ms / nfr)
            print("mode %d pipeline: %.3f ms/frame (%.1f frames/s), runs %s" % (
                mode, min(ms), 1e3 / min(ms), " ".join("%.3f" % v for v in ms)), flush=True)
        finally:
            fp.close()
        # kernel times: one lane, so that every kernel of the frame runs alone on its stream
        cfg1 = pipeline.make_pipeline_config(W, H, D, BS, mode, Q, K, lanes=1, max_points=20000, extractor=N.STEGER_IMPROVED)
        fp = pipeline.FramePipeline(cfg1, maps=maps, ctx=ctx)
        try:
            n1 = 4
            dL, dR = fp.upload(L[:n1]), fp.upload(R[:n1])
            fp.run_dev(dL, dR, n1)
            fp.set_timing(True)
            for rep in range(2):
                fp.run_dev(dL, dR, n1)
                out = []
                for g in GROUPS:
                    t, k = fp.kernel_time(g)
                    if k:
                        out.append("%s %.4f ms x%d" % (g, t / k, k // n1))
                print("mode %d per launch (alone): %s" % (mode, "  ".join(out)), flush=True)
        finally:
            fp.close()
        ctx.set_rectify_maps(0, maps[0], maps[1])
        ctx.set_rectify_maps(1, maps[2], maps[3])
        dc = pipeline.depth_config(D, BS, mode, Q)
        for _ in range(2):
            ctx.compute_depth(dc, base[0][0], base[0][1])
        lat = []
        for i in range(8):
            t0 = time.perf_counter()
            ctx.compute_depth(dc, base[i % 4][0], base[i % 4][1])  # host in, host out: ends in a device synchronise
            lat.append((time.perf_counter() - t0) * 1e3)
        print("mode %d compute_depth: median %.2f ms, min %.2f ms (host arrays in and out)" % (
            mode, float(np.median(lat)), min(lat)), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
