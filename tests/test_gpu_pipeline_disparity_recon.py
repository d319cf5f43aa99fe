"""The frame pipeline's disparity-domain reconstruction: the order test_improved_laser.py:112-207 runs for the
Improved / Hybrid extractors (left matcher -> disp / 16.0 -> extract_centerline -> reconstruct_from_disparity or
reconstruct_with_interpolation), with recon kinds DISPARITY and DISPARITY_MEDIAN reading each frame's int16 disparity.

For every case and frame the pipeline's 3D points equal, bit for bit, l3d_reconstruct on the same frame's fetched
points_2d and disp16 (float64) and ImprovedLaserReconstructorRef (after the float32 cast), in lane-per-frame, grouped
and CUDA-graph replay mode.  A numpy classifier labels every 2D point by the branch the restatement takes, and each
case asserts that every branch is taken a stated number of times."""
import ctypes as C
from collections import Counter

import numpy as np
import pytest
from numpy.lib.stride_tricks import sliding_window_view

from laser_3d_reconstruction_b200 import _native as N
from laser_3d_reconstruction_b200 import pipeline, synth
from laser_3d_reconstruction_b200.improved_reconstruction import ImprovedLaserReconstructor
from oracle import ref_ops

pytestmark = pytest.mark.gpu

CAP = 8000
EXTRACTORS = (N.EXTRACT_SIMPLE, N.STEGER_FAST, N.STEGER_IMPROVED, N.STEGER_HYBRID)
# (kind, window, min_disparity, far rig): "med" is the median disparity along the stripe, so that median windows often hold
# an even number of valid values; the far rig's baseline puts Z = 10 m at that median, so about half the points fail 0 < Z < 10
RECONS = ((N.RECON_DISPARITY, 3, "one", False), (N.RECON_DISPARITY, 3, "med", False),
          (N.RECON_DISPARITY_MEDIAN, 1, "one", True), (N.RECON_DISPARITY_MEDIAN, 3, "med", False),
          (N.RECON_DISPARITY_MEDIAN, 5, "one", True), (N.RECON_DISPARITY_MEDIAN, 9, "med", False))
BRANCHES = ("kept_odd", "kept_even", "border", "none_valid", "z", "invalid_centre")


def eq(a, b, what=""):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, "%s: shape %s vs %s" % (what, a.shape, b.shape)
    bad = np.argwhere(a != b)
    assert len(bad) == 0, "%s: %d/%d differ, first %s got %s want %s" % (
        what, len(bad), a.size, tuple(bad[0]), a[tuple(bad[0])], b[tuple(bad[0])])


def stripe_centre(W, H):
    """left-view stripe centre per row: a diagonal from past the left edge, through the columns x < D that the matcher
    never matches, to the bottom row at 0.72 W"""
    return -0.03 * W + 0.75 * W * np.arange(H) / (H - 1)


def scene(W, H, D, seed):
    """synth's textured pair with the diagonal stripe instead of the vertical one, painted into the right view at the
    scene's disparity"""
    left, right = synth.stereo_pair(W, H, D, seed, laser=False)
    xs = np.arange(W)[None, :]
    cx = stripe_centre(W, H)
    dc = synth.disparity_field(W, H, D)[np.arange(H), np.clip(np.rint(cx).astype(int), 0, W - 1)]
    colour = np.array([140.0, 255.0, 140.0], np.float32)

    def paint(img, centre):
        a = np.clip(3.0 * np.exp(-(xs - centre[:, None]) ** 2 / (2 * 2.5 ** 2)), 0, 1)[..., None]
        return np.rint(img.astype(np.float32) * (1 - a) + colour * a).astype(np.uint8)

    return paint(left, cx), paint(right, cx - dc)


def stripe_median_disparity(W, H, D):
    cx = stripe_centre(W, H)
    ok = (cx >= D) & (cx < W)
    return float(np.round(np.median(synth.disparity_field(W, H, D)[np.arange(H)[ok], np.rint(cx[ok]).astype(int)]), 2))


def batch(W, H, D, seeds):
    frames = [scene(W, H, D, s) for s in seeds]
    return np.stack([f[0] for f in frames]), np.stack([f[1] for f in frames])


def recon_for(W, H, D, kind, window, mind, far):
    """(ImprovedLaserReconstructor, its ReconParams) of one RECONS entry"""
    med = stripe_median_disparity(W, H, D)
    _, Q = synth.camera_model(W, H, baseline=10.0 * med / (0.8 * W) if far else 0.06)  # focal length 0.8 W
    ir = ImprovedLaserReconstructor(Q, verbose=False)
    return ir, ir.recon_params(kind, 1.0 if mind == "one" else med, window)


def classify(rp, fxb, xy, disp16, invalid16):
    """label of every 2D point by the branch ImprovedLaserReconstructorRef takes for it"""
    d = disp16.astype(np.float32) / 16.0
    H, W = d.shape
    px, py = np.rint(xy[:, 0]).astype(np.int64), np.rint(xy[:, 1]).astype(np.int64)
    mind = np.float32(rp.min_disparity)
    median = rp.kind == N.RECON_DISPARITY_MEDIAN
    hw = rp.window // 2 if median else 0
    lab = np.full(len(px), "", object)
    inb = (px >= hw) & (px < W - hw) & (py >= hw) & (py < H - hw)
    lab[~inb] = "border"
    i = np.nonzero(inb)[0]
    if not median:
        val = d[py[i], px[i]]
        low = val < mind
        lab[i[low]] = np.where(disp16[py[i], px[i]][low] == invalid16, "invalid_centre", "below_min")
        kept = np.full(len(i), "kept_odd", object)
    else:
        win = sliding_window_view(d, (rp.window, rp.window))[py[i] - hw, px[i] - hw].reshape(len(i), -1)
        good = win >= mind
        cnt = good.sum(1)
        low = cnt == 0
        lab[i[low]] = "none_valid"
        s = np.sort(np.where(good, win, np.float32(np.inf)), axis=1)
        k, r = np.maximum(cnt, 1), np.arange(len(i))
        val = np.where(k % 2 == 1, s[r, k // 2], (s[r, np.maximum(k // 2 - 1, 0)] + s[r, k // 2]) * np.float32(0.5))
        kept = np.where(cnt % 2 == 1, "kept_odd", "kept_even")
    with np.errstate(divide="ignore", invalid="ignore"):
        Z = fxb / val.astype(np.float64)
    rest = ~low
    lab[i[rest]] = np.where((Z > 0) & (Z < 10.0), kept, "z")[rest]
    return lab


def check_frames(ctx, fp, ir, rp, nframes, what):
    """every frame of the last run against the single-call path and the restatement; returns the branch counts"""
    assert fp.points_needed <= CAP
    ref = ref_ops.ImprovedLaserReconstructorRef(ir.Q)
    invalid16 = 16 * (fp.cfg.depth.left.minDisparity - 1)
    counts = Counter()
    out = []
    for f in range(nframes):
        got = fp.fetch(f)
        xy64, xyz64 = fp.fetch_points(f, want_2d=True)
        eq(got["points_2d"], xy64, "%s frame %d: points_2d" % (what, f))
        disp = got["disp16"].astype(np.float32) / 16.0
        eq(xyz64, ctx.reconstruct(rp, got["points_2d"], disp), "%s frame %d: pipeline vs l3d_reconstruct" % (what, f))
        pts = [tuple(p) for p in xy64]
        if rp.kind == N.RECON_DISPARITY:
            want = ref.reconstruct_from_disparity(pts, disp, rp.min_disparity)
        else:
            want = ref.reconstruct_with_interpolation(pts, disp, rp.window, rp.min_disparity)
        assert got["points_3d"].dtype == np.float32
        eq(got["points_3d"], want.reshape(-1, 3), "%s frame %d: pipeline vs ImprovedLaserReconstructorRef" % (what, f))
        lab = classify(rp, ir.fx * ir.baseline, xy64, got["disp16"], invalid16)
        assert "" not in set(lab)
        nkept = int(np.sum([s.startswith("kept") for s in lab]))
        assert nkept == len(xyz64) > 0, "%s frame %d: %d kept by the classifier, %d points" % (what, f, nkept, len(xyz64))
        counts.update(lab)
        out.append(dict(got, points_3d_f64=xyz64))
    return counts, out


def make_fp(ctx, W, H, D, bs, mode, depth, extractor, rp, lanes, maps=None):
    K, Q = synth.camera_model(W, H)
    cfg = pipeline.make_pipeline_config(W, H, D, bs, mode, Q, K, extractor=extractor, lanes=lanes, max_points=CAP,
                                        use_wls=depth == "wls", use_maps=maps is not None, recon=rp,
                                        mutated_left=depth == "mutated")
    return pipeline.FramePipeline(cfg, maps=maps, ctx=ctx)


def assert_branches(counts, minimum, what):
    short = {b: counts[b] for b in BRANCHES if counts[b] < minimum[b]}
    assert not short, "%s: branches taken too rarely %s (all counts %s)" % (what, short, dict(counts))


# every branch at least this often over one depth configuration's 4 extractors x 6 reconstructions x 2 frames
MIN_C1 = dict(kept_odd=2000, kept_even=100, border=20, none_valid=200, z=500, invalid_centre=50)


@pytest.mark.parametrize("depth", ["wls", "plain", "mutated"])
@pytest.mark.parametrize("mode", [0, 1, 2, 3])
def test_c1_kinds_windows_extractors(ctx, mode, depth):
    """c1 geometry (320x360, D 64, block 5), unrectified input so that the stripe reaches the image border; WLS on, the
    left matcher alone as constructed, and alone as createDisparityWLSFilter mutates it"""
    W, H, D, bs = 320, 360, 64, 5
    L, R = batch(W, H, D, (mode * 10 + 1, mode * 10 + 2))
    total = Counter()
    for ext in EXTRACTORS:
        xy_first = None
        for kind, window, mind, far in RECONS:
            ir, rp = recon_for(W, H, D, kind, window, mind, far)
            what = "mode %d %s extractor %d kind %d window %d" % (mode, depth, ext, kind, window)
            fp = make_fp(ctx, W, H, D, bs, mode, depth, ext, rp, lanes=1)
            try:
                counts = fp.run_host(L, R)
                c, out = check_frames(ctx, fp, ir, rp, len(L), what)
                assert list(counts) == [len(o["points_3d"]) for o in out]
            finally:
                fp.close()
            total += c
            xy = [o["points_2d"] for o in out]
            if xy_first is None:
                xy_first = xy
            for f in range(len(L)):  # the reconstruction does not feed back into the extraction
                eq(xy[f], xy_first[f], what + " frame %d: points_2d across recon kinds" % f)
    assert_branches(total, MIN_C1, "mode %d %s" % (mode, depth))


@pytest.mark.parametrize("mode,depth", [(1, "wls"), (1, "plain"), (0, "wls"), (0, "mutated")])
def test_lane_counts_and_grouped_mode_agree(ctx, mode, depth):
    """lanes 1 and 3 (lane per frame) and 14 (grouped: one cluster-fused aggregation per lane set, backs on the lanes'
    second streams): every bit of every frame identical, and each equal to the single-call path and the restatement"""
    W, H, D, bs = 320, 360, 64, 5
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    L, R = batch(W, H, D, range(20, 29))  # 9 frames: a full lane set of 7 and a ragged one with WLS
    for ext in (N.EXTRACT_SIMPLE, N.STEGER_IMPROVED):
        for kind, window, mind, far in (RECONS[0], RECONS[3]):
            ir, rp = recon_for(W, H, D, kind, window, mind, far)
            res = {}
            for lanes in (1, 3, 14):
                what = "mode %d %s extractor %d kind %d lanes %d" % (mode, depth, ext, kind, lanes)
                fp = make_fp(ctx, W, H, D, bs, mode, depth, ext, rp, lanes, maps)
                try:
                    dl, dr = fp.upload(L), fp.upload(R)
                    fp.run_dev(dl, dr, len(L))
                    _, res[lanes] = check_frames(ctx, fp, ir, rp, len(L), what)
                finally:
                    fp.close()
            for lanes in (3, 14):
                for f in range(len(L)):
                    for k in ("left_rect", "depth", "disp16", "points_2d", "points_3d", "points_3d_f64"):
                        eq(res[lanes][f][k], res[1][f][k], "lanes %d vs 1, %s frame %d (extractor %d kind %d)" % (lanes, k, f, ext, kind))


@pytest.mark.parametrize("recon", [RECONS[0], RECONS[3], RECONS[5]])
def test_graph_replay_host_buffers(ctx, recon):
    """set up as test_gpu_parity.py::test_pipeline_graph_replay_host_buffers: c1 geometry, 14 lanes, host buffers, the step
    repeated until it is replayed as a CUDA graph; replays give the direct launches' points, also for new content"""
    W, H, D, bs = 320, 360, 64, 5
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    ir, rp = recon_for(W, H, D, *recon)
    fp = make_fp(ctx, W, H, D, bs, 1, "wls", N.STEGER_IMPROVED, rp, 14, maps)
    try:
        frames = [scene(W, H, D, 90 + s) for s in range(14)]
        pL = pipeline.pinned_empty((14, H, W, 3), np.uint8); pR = pipeline.pinned_empty((14, H, W, 3), np.uint8)
        depth = pipeline.pinned_empty((14, H, W), np.float32); xyz = pipeline.pinned_empty((14, CAP, 3), np.float64)
        pL[:] = np.stack([f[0] for f in frames]); pR[:] = np.stack([f[1] for f in frames])
        counts0 = fp.run_host(pL, pR, depth, xyz)
        _, out0 = check_frames(ctx, fp, ir, rp, 14, "direct")
        x0 = [xyz[i, :counts0[i]].copy() for i in range(14)]
        for i in range(14):
            eq(x0[i], out0[i]["points_3d_f64"], "run_host xyz frame %d" % i)
        for _ in range(4):
            counts = fp.run_host(pL, pR, depth, xyz)
        assert fp.graph_replays >= 1
        assert list(counts) == list(counts0)
        _, out = check_frames(ctx, fp, ir, rp, 14, "replayed")
        for i in range(14):
            eq(xyz[i, :counts[i]], x0[i], "replayed xyz frame %d" % i)
            eq(out[i]["disp16"], out0[i]["disp16"], "replayed disp16 frame %d" % i)
        replays = fp.graph_replays
        pL[:] = pL[::-1].copy(); pR[:] = pR[::-1].copy()
        counts2 = fp.run_host(pL, pR, depth, xyz)
        assert fp.graph_replays == replays + 1
        assert list(counts2) == list(counts0)[::-1]
        check_frames(ctx, fp, ir, rp, 14, "replayed, new content")
        for i in range(14):
            eq(xyz[i, :counts2[i]], x0[13 - i], "replayed xyz, new content, frame %d" % i)
    finally:
        fp.close()


def test_c3_geometry(ctx):
    """1280x720, D 128, block 9, MODE_HH with WLS on 14 lanes (grouped, wavefront aggregation), as bench.py's c3 runs it"""
    W, H, D, bs = 1280, 720, 128, 9
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    L, R = batch(W, H, D, (3, 4, 5))
    total = Counter()
    for recon in (RECONS[0], RECONS[3], RECONS[4]):
        ir, rp = recon_for(W, H, D, *recon)
        fp = make_fp(ctx, W, H, D, bs, 1, "wls", N.STEGER_IMPROVED, rp, 14, maps)
        try:
            fp.run_host(L, R)
            c, _ = check_frames(ctx, fp, ir, rp, len(L), "c3 kind %d window %d" % (rp.kind, rp.window))
            total += c
        finally:
            fp.close()
    assert_branches(total, dict(kept_odd=500, kept_even=20, border=0, none_valid=20, z=20, invalid_centre=10), "c3")


def test_create_refuses_bad_median_window(ctx):
    """a DISPARITY_MEDIAN window that is not odd in [1, 9] fails at l3d_pipeline_create (L3D_ERR_ARG = -1); the same
    config under DEPTH is accepted"""
    W, H, D = 320, 360, 64
    K, Q = synth.camera_model(W, H)
    ir = ImprovedLaserReconstructor(Q, verbose=False)

    def create(rp):
        cfg = pipeline.make_pipeline_config(W, H, D, 5, 2, Q, K, lanes=1, max_points=CAP, recon=rp)
        h = C.c_void_p()
        rc = ctx.lib.l3d_pipeline_create(ctx.h, C.byref(cfg), C.byref(h))
        if rc == 0:
            ctx.lib.l3d_pipeline_destroy(h)
        return rc

    for w in (0, 2, 11):
        rp = ir.recon_params(N.RECON_DISPARITY_MEDIAN, 1.0, w)
        assert create(rp) == -1, w
        assert "median window" in ctx.lib.l3d_last_error(ctx.h).decode()
        rp.kind = N.RECON_DEPTH
        rp.K[:] = [float(v) for v in K.reshape(9)]
        assert create(rp) == 0, w
    for w in (1, 3, 5, 7, 9):
        assert create(ir.recon_params(N.RECON_DISPARITY_MEDIAN, 1.0, w)) == 0, w
