#!/usr/bin/env python
"""Frames/s of LaserReconstructionSystem.process_frames(frames=...) on side-by-side captures, where its host time goes,
and the frame pipeline's own rate next to it.

    python tools/process_frames_probe.py [--parent DIR] [--rounds 2] [--reps 2] [--json OUT]

For each geometry (config 1: 320x360 per eye, 64 disparities, block 5, SGBM_3WAY, no WLS, Simple extractor; config 3:
1280x720 per eye, 128 disparities, block 9, MODE_HH + WLS, FastSteger) and batch (112 and 448 frames) it reports
  process_frames   this tree's process_frames(frames=captures) (captures: one C-contiguous uint8 array)
  parent           the same call from the tree in --parent (another checkout of the project, built by this script),
                   run alternately with this tree's, round after round
  run_host         this tree's FramePipeline.run_host on the views split on the host beforehand, all frames in one call
  chunk sweep      run_captures_host over the frames in pieces of 28 / 56 / 112 / 224 frames (what CHUNK_FRAMES buys)
and, per process_frames call, its host time split into
  split            entry to the first pipeline call (the host split and stacking of the views where the version does it)
  pipeline         the run_host / run_captures_host calls (upload, GPU run, counts)
  fetch            the fetch calls (device -> host copies of images and points)
  convert          the rest: point tuples, NaN filter, the accumulated cloud
Each measurement runs in a process of its own (the two trees' packages share a name).  The captures are 8 synthetic
stereo pairs (synth.stereo_pair, laser line included) repeated; pageable host memory, as a caller's arrays are.
Prints the GPU's name and power limit and one JSON line per measurement.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GEOMS = {
    "c1": dict(W=320, H=360, D=64, BS=5, MODE=2, wls=False, extractor="simple"),
    "c3": dict(W=1280, H=720, D=128, BS=9, MODE=1, wls=True, extractor="steger"),
}
SWEEP = (28, 56, 112, 224)


def worker(root, geom, nframes, reps, sweep):
    sys.path.insert(0, root)
    import numpy as np
    import laser_3d_reconstruction_b200 as l3d
    from laser_3d_reconstruction_b200 import pipeline, synth
    from laser_3d_reconstruction_b200.system import LaserReconstructionSystem
    g = GEOMS[geom]
    W, H = g["W"], g["H"]
    K, _ = synth.camera_model(W, H)
    tmp = tempfile.mkdtemp(prefix="l3d_probe_")
    path = os.path.join(tmp, "stereo_calibration.json")
    with open(path, "w") as f:
        json.dump(dict(R=np.eye(3).tolist(), T=[[-0.06], [0.0], [0.0]], camera_matrix_left=K.tolist(),
                       dist_coeffs_left=[[0.01, -0.02, 0.0, 0.0, 0.0]], camera_matrix_right=K.tolist(),
                       dist_coeffs_right=[[-0.01, 0.015, 0.0, 0.0, 0.0]]), f)
    cam = l3d.SingleUSBStereoCameraManager(width=2 * W, height=H, calibration_file=path, num_disparities=g["D"],
                                           block_size=g["BS"], sgbm_mode=g["MODE"], use_wls=g["wls"], verbose=False)
    assert cam.initialize_offline()
    cfg = l3d.Config()
    cfg.LASER_EXTRACTOR_TYPE = g["extractor"]
    s = LaserReconstructionSystem(cfg, verbose=False)
    assert s.initialize(camera=cam)
    pairs = [synth.stereo_pair(W, H, g["D"], seed=k) for k in range(8)]
    base = np.stack([np.concatenate(p, axis=1) for p in pairs])
    caps = np.ascontiguousarray(base[np.arange(nframes) % len(pairs)])

    # host-time split of process_frames: wrap the calls both versions make
    FP = pipeline.FramePipeline
    acc = dict(pipeline=0.0, fetch=0.0, split=0.0)
    state = dict(entry=None, depth=0)

    def timed(fn, key):
        def w(*a, **k):
            if state["entry"] is not None and key == "pipeline":
                acc["split"] += time.perf_counter() - state["entry"]
                state["entry"] = None
            if state["depth"]:  # fetch() calls fetch_points(): count the outer call only
                return fn(*a, **k)
            state["depth"] += 1
            t = time.perf_counter()
            try:
                return fn(*a, **k)
            finally:
                acc[key] += time.perf_counter() - t
                state["depth"] -= 1
        return w

    for name, key in (("run_host", "pipeline"), ("run_captures_host", "pipeline"), ("fetch", "fetch"),
                      ("fetch_points", "fetch"), ("fetch_images", "fetch")):
        if hasattr(FP, name):
            setattr(FP, name, timed(getattr(FP, name), key))

    def call():
        s.point_cloud = []
        for k in acc:
            acc[k] = 0.0
        t = time.perf_counter()
        state["entry"] = t
        out = s.process_frames(frames=caps)
        total = time.perf_counter() - t
        assert len(out) == nframes
        return total, dict(acc), sum(len(o[2]) for o in out), len(s.point_cloud)

    call()  # warm-up: pipeline creation, scratch growth, first launches
    runs = [call() for _ in range(reps)]
    totals = [r[0] for r in runs]
    med = lambda xs: statistics.median(xs)
    res = dict(tree=root, geom=geom, frames=nframes, fps=[round(nframes / t, 1) for t in totals],
               ms_per_frame=round(1e3 * med(totals) / nframes, 3), points_2d=runs[-1][2], cloud=runs[-1][3])
    parts = {k: med([r[1][k] for r in runs]) for k in acc}
    parts["convert"] = med(totals) - sum(parts.values())
    res["host_ms_per_frame"] = {k: round(1e3 * v / nframes, 3) for k, v in parts.items()}
    if sweep:
        fp = s._pipe
        L = np.ascontiguousarray(caps[:, :, :W])
        R = np.ascontiguousarray(caps[:, :, W:])
        fp.run_host(L, R)
        t = time.perf_counter()
        for _ in range(reps):
            fp.run_host(L, R)
        res["run_host_fps"] = round(reps * nframes / (time.perf_counter() - t), 1)
        res["run_host_gpu_ms_per_frame"] = round(fp.last_ms / nframes, 4)
        res["chunk_sweep_fps"] = {}
        for k in SWEEP:
            pieces = [caps[c:c + k] for c in range(0, nframes, k)]
            for p in pieces:
                fp.run_captures_host(p, 0)
            t = time.perf_counter()
            for _ in range(reps):
                for p in pieces:
                    fp.run_captures_host(p, 0)
            res["chunk_sweep_fps"][k] = round(reps * nframes / (time.perf_counter() - t), 1)
    s.stop()
    print("RESULT " + json.dumps(res), flush=True)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = "nvidia-smi unavailable (%s)" % e
    return q


def run_worker(root, geom, n, reps, sweep):
    cmd = [sys.executable, os.path.abspath(__file__), "--worker", root, geom, str(n), str(reps)] + (["--sweep"] if sweep else [])
    p = subprocess.run(cmd, capture_output=True, text=True)
    for line in p.stdout.splitlines():
        if line.startswith("RESULT "):
            return json.loads(line[7:])
    raise RuntimeError("worker %s %s %d failed:\n%s\n%s" % (root, geom, n, p.stdout[-3000:], p.stderr[-3000:]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent", help="checkout of the parent commit (built here) to compare against")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--geoms", default="c1,c3")
    ap.add_argument("--frames", default="112,448")
    ap.add_argument("--json", help="also write every result to this file")
    ap.add_argument("--worker", nargs=4, metavar=("ROOT", "GEOM", "N", "REPS"), help=argparse.SUPPRESS)
    ap.add_argument("--sweep", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        root, geom, n, reps = a.worker
        return worker(root, geom, int(n), int(reps), a.sweep)
    trees = [("this", HERE)]
    if a.parent:
        parent = os.path.abspath(a.parent)
        subprocess.run([sys.executable, "-c", "import __graft_entry__ as g; g.build()"], cwd=parent, check=True)
        trees.append(("parent", parent))
    info = gpu_info()
    print("GPU (name, power limit, max SM clock): %s" % info, flush=True)
    results = []
    for geom in a.geoms.split(","):
        for n in [int(x) for x in a.frames.split(",")]:
            for rnd in range(a.rounds):
                for label, root in trees:
                    r = run_worker(root, geom, n, a.reps, sweep=(label == "this" and rnd == 0))
                    r.update(label=label, round=rnd, gpu=info)
                    results.append(r)
                    print(json.dumps(r), flush=True)
    print("\nsummary (median frames/s of process_frames(frames=...) over all rounds and reps):")
    for geom in a.geoms.split(","):
        for n in [int(x) for x in a.frames.split(",")]:
            row = []
            for label, _ in trees:
                fps = [f for r in results if r["geom"] == geom and r["frames"] == n and r["label"] == label for f in r["fps"]]
                row.append("%s %.1f" % (label, statistics.median(fps)))
            rh = [r for r in results if r["geom"] == geom and r["frames"] == n and "run_host_fps" in r]
            if rh:
                row.append("run_host %.1f (GPU %.3f ms/frame)" % (rh[0]["run_host_fps"], rh[0]["run_host_gpu_ms_per_frame"]))
                row.append("chunk sweep %s" % rh[0]["chunk_sweep_fps"])
            print("  %s, %d frames: %s" % (geom, n, "; ".join(row)))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(dict(gpu=info, results=results), f, indent=1)


if __name__ == "__main__":
    main()
