"""Frames/s of the frame pipeline with each reconstruction kind it runs after the depth path: DEPTH
(reconstruct_from_depth on the depth plane), DISPARITY and DISPARITY_MEDIAN (window 3, both on the frame's int16
disparity), at bench.py's c1 and c3 geometries, lane counts and extractors.  The three pipelines run alternately, in
rounds, on the same device-resident frames; each number is one step's CUDA-event time over its frames.  Prints the card,
its power limit and SM clock first.
Usage: python tools/recon_kind_probe.py [rounds] [steps per round]   (default 5 rounds of 3 steps)"""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from laser_3d_reconstruction_b200 import _native as N, pipeline, synth  # noqa: E402
from laser_3d_reconstruction_b200.improved_reconstruction import ImprovedLaserReconstructor  # noqa: E402

# name: (W, H, D, block, mode, use_wls, extractor, frames per step, lanes) as bench.py's configs
GEOMS = {"c1": (320, 360, 64, 5, 2, False, N.EXTRACT_SIMPLE, 448, 28),
         "c3": (1280, 720, 128, 9, 1, True, N.STEGER_IMPROVED, 112, 28)}


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks_throttle_reasons.active"
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True)
    except OSError:
        return "nvidia-smi unavailable"
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "nvidia-smi unavailable"


def main():
    rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    steps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    print("card: %s" % card(), flush=True)
    ctx = N.Context(0)
    for name, (W, H, D, BS, mode, wls, ext, nfr, lanes) in GEOMS.items():
        K, Q = synth.camera_model(W, H)
        maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
        base = [synth.stereo_pair(W, H, D, s) for s in range(8)]
        L = np.stack([base[i % 8][0] for i in range(nfr)])
        R = np.stack([base[i % 8][1] for i in range(nfr)])
        ir = ImprovedLaserReconstructor(Q, verbose=False)
        kinds = {"DEPTH": None, "DISPARITY": ir.recon_params(N.RECON_DISPARITY, 1.0),
                 "DISPARITY_MEDIAN": ir.recon_params(N.RECON_DISPARITY_MEDIAN, 1.0, 3)}
        fps, dev = {}, {}
        try:
            for k, rp in kinds.items():
                cfg = pipeline.make_pipeline_config(W, H, D, BS, mode, Q, K, extractor=ext, lanes=lanes, max_points=20000,
                                                    use_wls=wls, recon=rp)
                fps[k] = pipeline.FramePipeline(cfg, maps=maps, ctx=ctx)
                dev[k] = (fps[k].upload(L), fps[k].upload(R))
                for _ in range(4):  # scratch growth, then the CUDA-graph capture of a launch-bound step
                    fps[k].run_dev(*dev[k], nfr)
            ms = {k: [] for k in kinds}
            for _ in range(rounds):
                for k in kinds:
                    for _ in range(steps):
                        fps[k].run_dev(*dev[k], nfr)
                        ms[k].append(fps[k].last_ms)
            print("%s: %dx%d D %d block %d mode %d wls %d extractor %d, %d frames per step, %d lanes" % (
                name, W, H, D, BS, mode, wls, ext, nfr, lanes), flush=True)
            for k in kinds:
                f = [1e3 * nfr / v for v in ms[k]]
                print("  %-16s median %.1f frames/s (min %.1f, max %.1f over %d steps), points in frame 0: %d" % (
                    k, float(np.median(f)), min(f), max(f), len(f), len(fps[k].fetch_points(0))), flush=True)
        finally:
            for fp in fps.values():
                fp.close()
    ctx.close()


if __name__ == "__main__":
    main()
