#!/usr/bin/env python
"""bench.py -- the hot path of BASELINE.json on B200: frames/s and Gde/s of
rectify -> SGBM (left + right matcher) -> WLS -> depth -> laser centre line -> 3D,
frames sharded frame-wise over the GPUs.  Default workload: BASELINE config 3 (1280x720, 128 disparities, block 9,
MODE_HH + WLS + ImprovedSteger), the configuration the metric is quoted on; `--config c1|c2|c4|c5` select the others.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c3] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path over a batch of `--frames` synthetic frames per GPU (weak scaling; c5: the
4096-frame job split r::world, strong scaling).  Prints ONE JSON line on rank 0:
  value / ms_per_step : inputs resident in HBM, CUDA-event timed (l3d_pipeline_run_dev), max over ranks
  e2e                 : the same batch through the host-buffer C-ABI call (l3d_pipeline_run_host):
                        pinned H2D of every frame + D2H of depth maps and point clouds inside the timed region
  roofline            : one SGBM matcher run (cost volume + aggregation + WTA kernels) timed alone with CUDA
                        events on its stream, algorithmic bytes (SURVEY 8d) / duration vs the measured HBM peak
  latency_ms          : one frame at a time through the reference-facing calls (compute_depth, extract_centerline,
                        reconstruct_*): host arrays in, host arrays out
  cpu_baseline        : the reference's CPU path (cv2.StereoSGBM etc. through oracle/ref_ops.py) on a bounded
                        sample of the same frames, frame-parallel over the host cores (rank 0, N=1 only), and the
                        north_star acceptance list checked on one frame of the run (parity_check)
`--impl reference` times only that CPU path (all host threads, bounded sample per step).
`--dump-outputs DIR` writes what the device-resident arm computed in its last timed step as DIR/<name>.npy (see
dump_outputs); the inputs depend only on the arguments, so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

# one hardware work queue per stream (default 8): the frame pipeline drives 14 lane streams + 4 aggregation streams
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

MAX_POINTS = 20000
# BASELINE.json `configs` (SURVEY 8d "Configs -> concrete runs").  mode: cv2.STEREO_SGBM_MODE_* (1 = HH, 2 = SGBM_3WAY,
# the reference's own default); extractor / recon: what the reference's callers run at that configuration.
CONFIGS = {
    "c1": dict(W=320, H=360, D=64, BS=5, MODE=2, wls=False, extractor="simple", recon="depth", frames=448, lanes=28,
               cpu_frames_per_core=16,
               workload="c1: 320x360 per eye, 64 disparities, block 5, SGBM_3WAY (config.py defaults, as constructed) + "
                        "Simple HSV extractor + reconstruct_from_depth"),
    "c2": dict(W=320, H=360, D=64, BS=5, MODE=2, wls=True, extractor="fast", recon="plane_refraction", frames=448, lanes=28,
               cpu_frames_per_core=8,
               workload="c2: 320x360 per eye, 64 disparities, block 5, SGBM_3WAY (left+right matcher) + WLS(8000,1.5) + "
                        "FastSteger sigma 3 + reconstruct_laser_line with refraction correction (underwater config)"),
    "c3": dict(W=1280, H=720, D=128, BS=9, MODE=1, wls=True, extractor="improved", recon="depth", frames=112, lanes=28,
               cpu_frames_per_core=8,
               workload="c3: 1280x720 per eye, 128 disparities, block 9, SGBM MODE_HH (left+right matcher) + WLS(8000,1.5) "
                        "+ ImprovedSteger sigma 3 + reconstruct_from_depth"),
    "c4": dict(W=1920, H=1080, D=256, BS=11, MODE=1, wls=True, extractor="improved", recon="depth", frames=256, lanes=21,
               cpu_frames_per_core=1,
               workload="c4: 1920x1080 per eye, 256 disparities, block 11, SGBM MODE_HH (left+right matcher) + WLS(8000,1.5) "
                        "+ ImprovedSteger sigma 3 + reconstruct_from_depth, 256 frames per GPU and step streamed through "
                        "21 lanes of scratch volumes"),
    "c5": dict(W=1280, H=720, D=128, BS=9, MODE=1, wls=True, extractor="improved", recon="depth", frames=112, lanes=28,
               cpu_frames_per_core=8, job_frames=4096,
               workload="c5: 4096 frames of c3 (1280x720, 128 disparities, block 9, MODE_HH + WLS + ImprovedSteger) sharded "
                        "r::world over the GPUs, point clouds gathered to rank 0 by NCCL"),
}
W = H = D = BS = MODE = 0
CFG = None
WORKLOAD = ""


def select_config(name):
    global W, H, D, BS, MODE, CFG, WORKLOAD
    CFG = dict(CONFIGS[name], name=name)
    W, H, D, BS, MODE = CFG["W"], CFG["H"], CFG["D"], CFG["BS"], CFG["MODE"]
    WORKLOAD = CFG["workload"]


def sgbm_algorithmic_bytes():
    """SURVEY 8d: B_sgbm = (2 + 4*npasses)*N + 4*W*H bytes per matcher run; N = width1*H*D, npasses = 2 (HH), 1 (3WAY)."""
    n = (W - D) * H * D
    npasses = 2 if MODE == 1 else 1
    return (2 + 4 * npasses) * n + 4 * W * H


def pipeline_config(lanes):
    from laser_3d_reconstruction_b200 import _native as N
    from laser_3d_reconstruction_b200 import pipeline, synth
    K, Q = synth.camera_model(W, H)
    ex = {"simple": N.EXTRACT_SIMPLE, "fast": N.STEGER_FAST, "improved": N.STEGER_IMPROVED}[CFG["extractor"]]
    kw = {}
    if CFG["extractor"] == "simple":  # config.py:45-47 bounds
        kw = dict(bright_thr=200, hsv_lo=(50, 100, 180), hsv_hi=(70, 255, 255), min_area=50.0)
    cfg = pipeline.make_pipeline_config(W, H, D, BS, MODE, Q, K, extractor=ex, lanes=lanes, max_points=MAX_POINTS,
                                        use_wls=CFG["wls"], **kw)
    if CFG["recon"] == "plane_refraction":
        cfg.recon.kind = N.RECON_PLANE
        cfg.recon.plane[:] = [float(v) for v in synth.LASER_PLANE]
        cfg.recon.use_refraction = 1
    return cfg


def make_frames(n_distinct, nframes, seed0):
    from laser_3d_reconstruction_b200 import synth
    base = [synth.stereo_pair(W, H, D, seed0 + s) for s in range(n_distinct)]
    L = np.stack([base[i % n_distinct][0] for i in range(nframes)])
    R = np.stack([base[i % n_distinct][1] for i in range(nframes)])
    return L, R


# ----------------------------------------------------------------------------------------------
# CPU reference leg (oracle/ref_ops.py on the real cv2: TEST INFRASTRUCTURE used as a timed baseline)
# ----------------------------------------------------------------------------------------------
_CPU = {}


def _cpu_init(maps, K, Q):
    import cv2
    cv2.setNumThreads(1)  # MODE_HH is single-threaded inside OpenCV anyway: parallelise over frames
    _CPU.update(maps=maps, K=K, Q=Q)


def _cpu_frame(pair):
    from laser_3d_reconstruction_b200 import synth
    from oracle import ref_ops
    left, right = pair
    rect, depth = ref_ops.depth_path(left, right, _CPU["maps"], D, BS, MODE, _CPU["Q"], use_wls=CFG["wls"])
    if CFG["extractor"] == "simple":
        pts = ref_ops.simple_extract(rect, (50, 100, 180), (70, 255, 255), 200, 50)
    elif CFG["extractor"] == "fast":
        pts = ref_ops.fast_steger_extract(rect, loop=True)
    else:
        pts = ref_ops.improved_steger_extract(rect, loop=True)  # per-pixel np.linalg.eig, as the reference does
    rec = ref_ops.ReconstructorRef(_CPU["K"], synth.LASER_PLANE, CFG["recon"] == "plane_refraction")
    xyz = rec.reconstruct_laser_line(pts) if CFG["recon"] == "plane_refraction" else rec.reconstruct_from_depth(pts, depth)
    return int(len(xyz))


class CpuPath:
    def __init__(self, max_workers=32):
        import multiprocessing as mp
        from laser_3d_reconstruction_b200 import synth
        try:
            ncpu = len(os.sched_getaffinity(0))
        except AttributeError:
            ncpu = os.cpu_count() or 1
        self.cores = max(1, min(ncpu, max_workers))  # each worker holds ~0.5 GB of OpenCV cost volumes
        K, Q = synth.camera_model(W, H)
        maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
        self.pool = mp.get_context("fork").Pool(self.cores, initializer=_cpu_init, initargs=(maps, K, Q))  # CFG is inherited

    def run(self, pairs):
        t0 = time.perf_counter()
        counts = self.pool.map(_cpu_frame, pairs, chunksize=1)
        return time.perf_counter() - t0, counts

    def close(self):
        self.pool.close()
        self.pool.join()


def bench_config(nfr, n_distinct, lanes, world):
    """the `config` object both arms print (same keys, so the driver's same_config check compares like with like)"""
    return {"workload": WORKLOAD, "name": CFG["name"], "frames_per_step_per_gpu": nfr, "distinct_frames": n_distinct,
            "lanes": lanes,
            "sharding": "frame-wise r::world, no collective on the hot path; NCCL gather of point clouds to rank 0"
                        " per step when N>1",
            "l2": "inputs plus %.0f MB of C/S cost volumes per matcher run exceed the 126 MB L2"
                  % (4.0 * (W - D) * H * D / 1e6),
            "gde_definition": "W*H*D per frame, counted once although two matchers run (SURVEY 8d)"}


def run_reference(args, rank):
    """`--impl reference`: the reference's own CPU implementation of the path, all host threads of ONE host (rank 0;
    at N > 1 the other ranks exit -- the per-N ratio against it is therefore scaling, not a per-GPU speed-up)."""
    if rank != 0:
        return
    from laser_3d_reconstruction_b200 import synth
    cpu = CpuPath()
    nfr = cpu.cores  # one frame per worker and step: a bounded sample of the workload
    base = [synth.stereo_pair(W, H, D, s) for s in range(min(nfr, 8))]
    pairs = [base[i % len(base)] for i in range(nfr)]
    for _ in range(args.warmup):
        cpu.run(pairs[:max(1, min(nfr, cpu.cores))])
    t = 0.0
    for _ in range(args.steps):
        dt, counts = cpu.run(pairs)
        t += dt
    cpu.close()
    fps = nfr * args.steps / t
    sample = "%d frames/step (one per worker), %d steps" % (nfr, args.steps)
    cfg = bench_config(args.frames or CFG["frames"], min(args.distinct, args.frames or CFG["frames"]),
                       args.lanes or CFG["lanes"], 1)
    out = {
        "impl": "reference", "metric": "frames_per_s", "value": fps, "unit": "frames/s", "gde_per_s": fps * W * H * D / 1e9,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16", "data": "synthetic",
        "config": cfg,   # exactly the GPU arm's object: the sample the CPU arm times per step is stated below, not here
        "reference_frames_per_step": nfr,
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cpu.cores, "kind": "port", "sample": sample,
                         "note": "cv2 %s StereoSGBM/remap/cvtColor (the binary the reference calls) driven by "
                                 "oracle/ref_ops.py; WLS = oracle C restatement (cv2.ximgproc absent); Steger = "
                                 "per-pixel np.linalg.eig loop as in the reference; one host's cores whatever N is"
                                 % __import__("cv2").__version__},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


# ----------------------------------------------------------------------------------------------
# clocks sampler
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.samples = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [s for (t, s) in self.samples if t0 <= t <= t1] or [s for (_, s) in self.samples[-3:]]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except (ValueError, IndexError):
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def parity_check(ctx, fp, frame, pair, maps, K, Q):
    """north_star's acceptance list on one frame of the run: GPU results (frame slot `frame` of the pipeline's last run
    and the single-call matcher pair) against cv2 / the reference restatement.  Executes oracle/ (checker only)."""
    import cv2
    from laser_3d_reconstruction_b200 import _native as N
    from laser_3d_reconstruction_b200 import synth
    from oracle import ref_ops
    left, right = pair
    got = fp.fetch(frame)
    wrect, wdepth, aux = ref_ops.depth_path(left, right, maps, D, BS, MODE, Q, use_wls=CFG["wls"], want_all=True)
    res = {"frame": int(frame), "rectified_equal_cv2_remap": bool(np.array_equal(got["left_rect"], wrect))}
    base, mut, rgt = ref_ops.sgbm_param_sets(D, BS, MODE)
    if CFG["wls"]:
        dl, dr = ctx.sgbm_compute_pair(N.SgbmParams(**mut), N.SgbmParams(**rgt), aux["lg"], aux["rg"])
        res["disparity_left_equal_cv2"] = bool(np.array_equal(dl, aux["dl"]))
        res["disparity_right_equal_cv2"] = bool(np.array_equal(dr, aux["dr"]))
        diff = np.abs(got["disp16"].astype(np.int32) - aux["df"].astype(np.int32))
        res["wls_within_1lsb_frac"] = float((diff <= 1).mean())
        res["wls_note"] = "against the oracle's restatement of cv2.ximgproc (parity unpinned: ximgproc is not installed)"
    else:
        res["disparity_left_equal_cv2"] = bool(np.array_equal(got["disp16"], aux["dl"]))
    if CFG["extractor"] == "simple":
        wp = np.array(ref_ops.simple_extract(wrect, (50, 100, 180), (70, 255, 255), 200, 50), np.float64).reshape(-1, 2)
        res["simple_points_equal"] = bool(wp.shape == got["points_2d"].shape and np.array_equal(wp, got["points_2d"]))
    else:
        fn = ref_ops.fast_steger_extract if CFG["extractor"] == "fast" else ref_ops.improved_steger_extract
        wp = np.array(fn(wrect), np.float64).reshape(-1, 2)
        gp = got["points_2d"].astype(np.float64)
        if len(wp) and len(gp):
            from scipy.spatial import cKDTree
            d1, d2 = cKDTree(wp).query(gp)[0], cKDTree(gp).query(wp)[0]
            res["steger_agreement_frac_0.01px"] = float(min((d1 <= 0.01).mean(), (d2 <= 0.01).mean()))
        else:
            res["steger_agreement_frac_0.01px"] = float(len(wp) == len(gp))
    rec = ref_ops.ReconstructorRef(K, synth.LASER_PLANE, CFG["recon"] == "plane_refraction")
    pts = [tuple(q) for q in got["points_2d"].astype(np.float64)]
    w3 = (rec.reconstruct_laser_line(pts) if CFG["recon"] == "plane_refraction"
          else rec.reconstruct_from_depth(pts, got["depth"])).reshape(-1, 3)
    g3 = got["points_3d"]
    res["points_3d"] = int(len(g3))
    res["points_3d_max_rel_err"] = (float(np.max(np.abs(g3 - w3) / np.maximum(np.abs(w3), 1e-12)))
                                    if g3.shape == w3.shape and len(g3) else (0.0 if g3.shape == w3.shape else None))
    res["ok"] = bool(res["rectified_equal_cv2_remap"] and res.get("disparity_left_equal_cv2", True)
                     and res.get("disparity_right_equal_cv2", True) and res.get("wls_within_1lsb_frac", 1.0) >= 0.999
                     and res.get("simple_points_equal", True) and res.get("steger_agreement_frac_0.01px", 1.0) >= 0.999
                     and res["points_3d_max_rel_err"] is not None and res["points_3d_max_rel_err"] <= 1e-5)
    return res


def single_frame_latency(ctx, pair, maps, K, Q, reps=10):
    """One frame at a time through the reference-facing calls (host arrays in and out): compute_depth =
    SingleUSBStereoCameraManager.get_frames without the capture, then extract_centerline, then reconstruct_*."""
    import laser_3d_reconstruction_b200 as l3d
    from laser_3d_reconstruction_b200 import pipeline, synth
    ctx.set_rectify_maps(0, maps[0], maps[1])
    ctx.set_rectify_maps(1, maps[2], maps[3])
    dcfg = pipeline.depth_config(D, BS, MODE, Q, use_wls=CFG["wls"])
    if CFG["extractor"] == "simple":
        ex = l3d.SimpleLaserExtractor(hsv_lower=[50, 100, 180], hsv_upper=[70, 255, 255], brightness_threshold=200, min_area=50,
                                      verbose=False)
    elif CFG["extractor"] == "fast":
        ex = l3d.FastStegerExtractor(sigma=3.0, verbose=False)
    else:
        ex = l3d.ImprovedStegerExtractor(sigma=3.0, verbose=False)
    rec = l3d.Reconstructor(K, synth.LASER_PLANE, CFG["recon"] == "plane_refraction")
    t = {"compute_depth": [], "extract_centerline": [], "reconstruct": []}
    for i in range(reps + 2):
        t0 = time.perf_counter()
        rect, depth = ctx.compute_depth(dcfg, pair[0], pair[1])
        t1 = time.perf_counter()
        pts = ex.extract_centerline(rect)
        t2 = time.perf_counter()
        if CFG["recon"] == "plane_refraction":
            rec.reconstruct_laser_line(pts)
        else:
            rec.reconstruct_from_depth(pts, depth)
        t3 = time.perf_counter()
        if i >= 2:
            t["compute_depth"].append(t1 - t0); t["extract_centerline"].append(t2 - t1); t["reconstruct"].append(t3 - t2)
    out = {k: 1e3 * float(np.median(v)) for k, v in t.items()}
    out["frame"] = sum(out.values())
    return out


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, fp, counts):
    """`--dump-outputs`: the results of the pipeline's last run, as a caller of the timed path receives them, in float32
    (images, depth, disparity, Steger centres) or float64 (counts, Simple centres, 3D points) .npy files under out_dir:
      counts.npy                  3D points of every frame slot of the run
      frameNNN_<key>.npy          FramePipeline.fetch(NNN): left_rect, depth, disp16 (int16 fixed point x16 as stored),
                                  points_2d, points_3d
    The full per-frame outputs of a whole step exceed 64 MB at the larger configs, so the frame slots are a fixed seeded
    sample (the same for every run with the same arguments), as many as fit in 64 MB.  A c5 step runs the job as several
    pipeline runs (chunks of --frames frames, all on the same resident inputs); the pipeline keeps only the last one, so
    for c5 the files hold that last chunk, not the whole job."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(counts)
    per_frame = (3 + 1 + 1) * 4 * W * H + (2 + 3) * 8 * MAX_POINTS + 5 * 128  # upper bound, .npy headers included
    k = max(1, min(n, (DUMP_BYTES - 8 * n - 128) // per_frame))
    slots = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
    np.save(os.path.join(out_dir, "counts.npy"), np.asarray(counts, np.float64))
    for f in slots:
        for key, a in fp.fetch(int(f)).items():
            a = a if a.dtype in (np.float32, np.float64) else a.astype(np.float32)
            np.save(os.path.join(out_dir, "frame%03d_%s.npy" % (f, key)), a)


def run_gpu(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from laser_3d_reconstruction_b200 import _native as N
    from laser_3d_reconstruction_b200 import pipeline, sharding, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    nfr = args.frames or CFG["frames"]      # frames per pipeline run (chunk) and GPU
    lanes = args.lanes or CFG["lanes"]
    strong = "job_frames" in CFG             # c5: a fixed job of 4096 frames, rank r takes frames r::world
    job = CFG.get("job_frames", nfr * world)
    K, Q = synth.camera_model(W, H)
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    if strong:
        mine_all = sharding.shard_frames(job, rank, world)
        chunks = [mine_all[i:i + nfr] for i in range(0, len(mine_all), nfr)]
    else:
        mine_all = sharding.shard_frames(nfr * world, rank, world)
        chunks = [mine_all]
    n_distinct = min(args.distinct, nfr)
    L, R = make_frames(n_distinct, nfr, seed0=1000 * rank)
    ctx = N.Context(local_rank)
    cfg = pipeline_config(lanes)
    fp = pipeline.FramePipeline(cfg, maps=maps, ctx=ctx)
    dL, dR = fp.upload(L), fp.upload(R)
    pL = pipeline.pinned_empty(L.shape, np.uint8)
    pR = pipeline.pinned_empty(R.shape, np.uint8)
    pL[:] = L
    pR[:] = R
    depth_h = pipeline.pinned_empty((nfr, H, W), np.float32)
    xyz_h = pipeline.pinned_empty((nfr, MAX_POINTS, 3), np.float64)

    def gather(ids, counts):
        """NCCL gather of the per-frame point clouds to rank 0 (the only exchange, off the hot path)."""
        if world == 1:
            return None
        table = torch.empty((max(int(np.sum(counts)), 1), 4), dtype=torch.float64, device=dev)
        rows = fp.pack_points_dev(ids, table.data_ptr())  # device-side pack; nothing goes through the host
        return sharding.gather_point_clouds(table[:rows], device=dev, to_host=False)  # stays on rank 0's GPU

    def step_dev():
        ms, counts = 0.0, None
        for ids in chunks:  # one chunk unless the job is larger than the resident batch (c5)
            counts = fp.run_dev(dL, dR, len(ids))
            ms += fp.last_ms
            gather(ids, counts)
        return counts, ms

    def step_host():
        ms, counts = 0.0, None
        for ids in chunks:
            n = len(ids)
            counts = fp.run_host(pL[:n], pR[:n], depth_h[:n], xyz_h[:n])
            ms += fp.last_ms
        return counts, ms

    # ---- device-resident arm -----------------------------------------------------------------
    warm = max(args.warmup, 3)
    for _ in range(warm):
        counts, _ = step_dev()
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    l0 = fp.launches
    t0 = time.perf_counter()
    dev_ms = 0.0
    for _ in range(args.steps):
        counts, ms = step_dev()
        dev_ms += ms
    barrier()
    t1 = time.perf_counter()
    wall_ms = (t1 - t0) * 1e3
    launches = fp.launches - l0
    clocks = sampler.stop(t0, t1) if sampler else None
    # a step's duration = CUDA-event time of the batch (first enqueue -> last lane done) + the gather's wall time
    # for N > 1; the wall clock over the K steps bounds it from above, so use the wall clock when gathering.
    el = torch.tensor([wall_ms if world > 1 else dev_ms, wall_ms], dtype=torch.float64, device=dev)
    nl = torch.tensor([launches], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
        dist.all_reduce(nl, op=dist.ReduceOp.SUM)
    elapsed_ms, wall_max = float(el[0]), float(el[1])
    launches = int(nl[0])  # kernels of libl3d.so launched inside the timed region, summed over ranks
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, fp, counts)

    # ---- end-to-end arm (host buffers through the C ABI) ----------------------------------------
    for _ in range(2):
        step_host()
    barrier()
    t0 = time.perf_counter()
    e2e_ms = 0.0
    for _ in range(args.steps):
        counts_h, ms = step_host()
        e2e_ms += ms
    barrier()
    e2e_wall = (time.perf_counter() - t0) * 1e3
    ee = torch.tensor([e2e_wall], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ee, op=dist.ReduceOp.MAX)
    e2e_elapsed = float(ee[0])
    assert list(counts_h) == list(counts), "host-buffer and device-resident runs disagree"
    frames_step_rank = sum(len(c) for c in chunks)
    per_frame_in = 2 * W * H * 3
    per_frame_out = W * H * 4 + MAX_POINTS * 24 + 8
    h2d = int(frames_step_rank * per_frame_in)
    d2h = int(frames_step_rank * per_frame_out)

    total_frames = (job if strong else nfr * world) * args.steps
    fps = total_frames / (elapsed_ms / 1e3)
    e2e_fps = total_frames / (e2e_elapsed / 1e3)
    config = bench_config(nfr, n_distinct, lanes, world)
    if strong:
        config["job_frames"] = job
        config["chunks_per_step_per_gpu"] = len(chunks)
    out = {
        "metric": "frames_per_s", "value": fps, "unit": "frames/s", "gde_per_s": fps * W * H * D / 1e9,
        "n_gpus": world, "steps": args.steps, "warmup": warm, "ms_per_step": elapsed_ms / args.steps,
        "wall_ms_per_step": wall_max / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak",
        "vs_baseline": None, "dtype": "int16", "data": "synthetic",
        "config": config,
        "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_elapsed / args.steps},
        "gpu_launches": int(launches),
        "points_per_frame": float(np.mean(counts)),
    }
    if clocks is not None:
        out["clocks"] = clocks

    # ---- roofline leg: the SGBM kernels timed alone (lanes chained, nothing overlaps them) ----------
    if rank == 0:
        fp1 = pipeline.FramePipeline(pipeline_config(lanes), maps=maps, ctx=ctx)
        nr = min(nfr, 14)
        for _ in range(2):
            fp1.run_dev(dL, dR, nr)
        fp1.set_timing(True)
        fp1.run_dev(dL, dR, nr)
        names = ["sgbm_cost", "sgbm_scan_k0", "sgbm_vgroup_down", "sgbm_vgroup_up", "sgbm_vwave_down", "sgbm_vwave_up", "sgbm_wta", "wls"] + \
                ["sgbm_scan_k%d" % kk for kk in range(1, 8)]
        groups = {}
        for g in names:
            t, k = fp1.kernel_time(g)
            if k:
                groups[g] = {"ms_total": t, "timed_regions": k}
        fp1.set_timing(False)
        runs = (2 if CFG["wls"] else 1) * nr  # left (+ right) matcher per frame
        sgbm_ms = sum(v["ms_total"] for g, v in groups.items() if g.startswith("sgbm_")) / runs
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except (OSError, ValueError):
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        achieved = sgbm_algorithmic_bytes() / (sgbm_ms * 1e-3) / 1e9
        traffic = None  # DRAM bytes of the same kernels from the committed ncu --set full capture (static, per config)
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(
                "sgbm_run_dram_bytes" if CFG["name"] in ("c3", "c5") else "sgbm_run_dram_bytes_" + CFG["name"])
        except (OSError, ValueError, KeyError):
            pass
        out["roofline"] = {
            "bound": "hbm", "kernel": "sgbm matcher run = cost volume (one pixel-cost pass feeds both matchers' volumes) + "
                                      "aggregation (config 3: two wavefront passes of four paths each, WTA fused into the second; other "
                                      "geometries: horizontal pair + cluster-fused previous-row passes) + WTA",
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "peak_source": "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6650 GB/s",
            "algorithmic_bytes_per_run": sgbm_algorithmic_bytes(), "ms_per_run": sgbm_ms, "traffic": traffic,
            "traffic_source": "static: profiles/traffic.json (ncu --set full capture of this build's kernels), not "
                              "re-measured in this run",
            "how": "CUDA events on the launching streams around every kernel group; lanes chained so each timed kernel "
                   "runs alone; %d frames = %d matcher runs; launches that serve several runs (the shared pixel-cost pass, "
                   "the cluster-fused aggregation of a lane set) are divided by the runs they process" % (nr, runs),
            "groups_ms_per_run": {g: v["ms_total"] / runs for g, v in groups.items() if g.startswith("sgbm_")},
            "wls_ms_per_frame": groups.get("wls", {"ms_total": 0.0})["ms_total"] / nr,
        }
        fp1.close()
        # the same pipeline object again after the timing run, for the parity check below
        fp.run_dev(dL, dR, min(nfr, len(chunks[-1])))
        out["latency_ms"] = single_frame_latency(ctx, (L[0], R[0]), maps, K, Q)

    # ---- CPU baseline leg (rank 0, N = 1 only): bounded sample ----------------------------------
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = CpuPath()
        ns = CFG["cpu_frames_per_core"] * cpu.cores  # ~10-30 s of CPU work
        pairs = [(L[i % nfr], R[i % nfr]) for i in range(ns)]
        dt, ccounts = cpu.run(pairs)
        cpu.close()
        out["cpu_baseline"] = {"value": ns / dt, "unit": "frames/s", "cores": cpu.cores, "kind": "port",
                               "sample": "%d frames of the same workload, frame-parallel over %d worker processes, %.1f s"
                                         % (ns, cpu.cores, dt),
                               "parity_check": parity_check(ctx, fp, 0, (L[0], R[0]), maps, K, Q)}
    if rank == 0:
        print(json.dumps(out), flush=True)
    fp.close()
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS), help="BASELINE.json configuration (default: the one the metric is quoted on)")
    ap.add_argument("--frames", type=int, default=0, help="frames per step per GPU (default per config; a multiple of the 7-frame lane set)")
    ap.add_argument("--distinct", type=int, default=8, help="distinct synthetic frames rendered per rank")
    ap.add_argument("--lanes", type=int, default=0, help="frames in flight per GPU (streams; default per config: 28 = four lane sets of 7 frames)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the outputs of the last timed step (rank 0, GPU arm) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs; the reference arm keeps none")
    select_config(args.config)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world == 1 and args.gpus > 1:
        # convenience: re-launch under torchrun, one process per GPU
        import socket
        with socket.socket() as s:
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    run_gpu(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
