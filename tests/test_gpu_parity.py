"""Parity of the sm_100a kernels (through the C ABI, via ctypes) against cv2 -- the library the
reference calls -- and against the oracle restatement for intermediates cv2 never exposes.
Bit-exact for integer stages; stated tolerances for WLS (unpinned), Steger centres and 3D points."""
import ctypes as C
import math

import cv2
import numpy as np
import pytest

from laser_3d_reconstruction_b200 import _native as N
from laser_3d_reconstruction_b200 import pipeline, synth
from oracle import cref, ref_ops

pytestmark = pytest.mark.gpu


def gray_pair(W, H, D, seed, quant=0):
    l, r = synth.stereo_pair(W, H, D, seed)
    lg, rg = cv2.cvtColor(l, cv2.COLOR_BGR2GRAY), cv2.cvtColor(r, cv2.COLOR_BGR2GRAY)
    if quant:
        lg = (lg // quant * quant).astype(np.uint8)
        rg = (rg // quant * quant).astype(np.uint8)
    return lg, rg


def eq(a, b, what=""):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, "%s: shape %s vs %s" % (what, a.shape, b.shape)
    bad = np.argwhere(a != b)
    assert len(bad) == 0, "%s: %d/%d differ, first %s got %s want %s" % (
        what, len(bad), a.size, tuple(bad[0]), a[tuple(bad[0])], b[tuple(bad[0])])


# ---- K1 remap + gray -----------------------------------------------------------------------
@pytest.mark.parametrize("case", range(4))
def test_remap_gray(ctx, case):
    rng = np.random.default_rng(case)
    H, W = (53, 97) if case == 0 else (240, 320)
    src = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    mx = (rng.random((H, W)) * (W + 8) - 4).astype(np.float32)  # includes out-of-range taps (border 0)
    my = (rng.random((H, W)) * (H + 8) - 4).astype(np.float32)
    if case == 1:
        mx = (np.round(mx * 64) / 64).astype(np.float32)
        my = (np.round(my * 64) / 64).astype(np.float32)
    if case == 3:
        mx, my = synth.warp_maps(W, H, 2)
    ctx.set_rectify_maps(0, mx, my)
    rect, gray = ctx.remap_gray(0, src, (H, W))
    want = cv2.remap(src, mx, my, cv2.INTER_LINEAR)
    eq(rect, want, "remap")
    eq(gray, cv2.cvtColor(want, cv2.COLOR_BGR2GRAY), "gray")


def test_remap_noncontiguous_view_and_real_pair(ctx, golden_real):
    g = golden_real
    size = (320, 240)
    R1, R2, P1, P2, Q, _, _ = cv2.stereoRectify(g["K_left"], g["dist_left"], g["K_right"], g["dist_right"], size,
                                                g["R"], g["T"], flags=cv2.CALIB_ZERO_DISPARITY, alpha=0)
    mlx, mly = cv2.initUndistortRectifyMap(g["K_left"], g["dist_left"], R1, P1, size, cv2.CV_32FC1)
    mrx, mry = cv2.initUndistortRectifyMap(g["K_right"], g["dist_right"], R2, P2, size, cv2.CV_32FC1)
    ctx.set_rectify_maps(0, mlx, mly)
    ctx.set_rectify_maps(1, mrx, mry)
    for tag in ("a", "b"):
        frame = g["frame_" + tag]
        l, r = frame[:, :320], frame[:, 320:]  # _split_frame views
        eq(ctx.remap_gray(0, l, (240, 320))[0], g["lrect_" + tag], "left rect")
        eq(ctx.remap_gray(1, r, (240, 320))[0], g["rrect_" + tag], "right rect")


def colour_cube(r0, r1):
    """all 2^16 (B, G) combinations for every R in [r0, r1): slices of the full 2^24 colour cube"""
    b, g = np.meshgrid(np.arange(256, dtype=np.uint8), np.arange(256, dtype=np.uint8), indexing="ij")
    planes = [np.stack([b, g, np.full_like(b, r)], -1) for r in range(r0, r1)]
    return np.ascontiguousarray(np.concatenate(planes, 0))


def test_colour_arithmetic_full_cube(ctx):
    """SURVEY 8c pin (iii): BGR->gray, BGR->HSV and inRange over ALL 2^24 colours, on the GPU, against cv2 -- gray through
    l3d_bgr2gray, HSV through l3d_colour_mask with range boxes that cut every channel (incl. the hue wrap at 0 / 179 and
    the S / V extremes), bit-exact."""
    boxes = [((50, 100, 180), (70, 255, 255)), ((40, 50, 100), (80, 255, 255)), ((0, 0, 0), (0, 255, 255)),
             ((179, 1, 1), (179, 255, 255)), ((0, 0, 0), (179, 0, 255)), ((90, 128, 0), (150, 129, 127)),
             ((10, 254, 254), (170, 255, 255)), ((0, 1, 1), (179, 254, 254))]
    for r0 in range(0, 256, 32):
        img = colour_cube(r0, r0 + 32)  # 8192 x 256 x 3
        eq(ctx.bgr2gray(img), cv2.cvtColor(img, cv2.COLOR_BGR2GRAY), "gray, R in [%d, %d)" % (r0, r0 + 32))
        hsv = cv2.cvtColor(img, cv2.COLOR_BGR2HSV)
        for lo, hi in boxes:
            eq(ctx.colour_mask(img, lo, hi), cv2.inRange(hsv, np.array(lo, np.uint8), np.array(hi, np.uint8)),
               "inRange(HSV) %s-%s, R in [%d, %d)" % (lo, hi, r0, r0 + 32))
        gray = cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)
        want = cv2.inRange(hsv, np.array(boxes[0][0], np.uint8), np.array(boxes[0][1], np.uint8)) & ((gray > 200) * np.uint8(255))
        eq(ctx.colour_mask(img, boxes[0][0], boxes[0][1], 200), want, "config.py colour + brightness mask")


def test_sgbm_more_real_pairs(ctx, golden_real, golden_real_more):
    """Four more of the reference's 28 calibration pairs (tests/golden/real_pair_[c-f].npz from the REAL camera class): the
    rectified views (CRC32 of cv2.remap's output), the as-constructed 3WAY matcher's int16 disparity and the depth image."""
    import zlib
    g = golden_real
    more = golden_real_more
    size = (320, 240)
    R1, R2, P1, P2, Q, _, _ = cv2.stereoRectify(g["K_left"], g["dist_left"], g["K_right"], g["dist_right"], size,
                                                g["R"], g["T"], flags=cv2.CALIB_ZERO_DISPARITY, alpha=0)
    mlx, mly = cv2.initUndistortRectifyMap(g["K_left"], g["dist_left"], R1, P1, size, cv2.CV_32FC1)
    mrx, mry = cv2.initUndistortRectifyMap(g["K_right"], g["dist_right"], R2, P2, size, cv2.CV_32FC1)
    ctx.set_rectify_maps(0, mlx, mly)
    ctx.set_rectify_maps(1, mrx, mry)
    base, _, _ = ref_ops.sgbm_param_sets(64, 5, 2)
    crc = lambda a: zlib.crc32(np.ascontiguousarray(a).tobytes())
    for tag in ("c", "d", "e", "f"):
        frame = more["frame_" + tag]
        lrect, lg = ctx.remap_gray(0, frame[:, :320], (240, 320))
        rrect, rg = ctx.remap_gray(1, frame[:, 320:], (240, 320))
        assert crc(lrect) == int(more["lrect_crc_" + tag]) and crc(rrect) == int(more["rrect_crc_" + tag]), tag
        d16 = ctx.sgbm_compute(N.SgbmParams(**base), lg, rg)
        eq(d16, more["disp16_" + tag], "real pair " + tag)
        assert crc(ctx.disp_to_depth(d16, Q)) == int(more["depth_crc_" + tag]), tag


# ---- K2 SGBM -------------------------------------------------------------------------------
SMALL = [(96, 48, 16, 3), (130, 50, 32, 5), (200, 64, 64, 9), (300, 56, 128, 7), (400, 48, 256, 11), (180, 52, 96, 5),
         (120, 50, 48, 3)]


@pytest.mark.parametrize("mode", [0, 1, 2, 3])  # 3 = MODE_HH4
@pytest.mark.parametrize("shape", SMALL)
def test_sgbm_small_all_roles(ctx, mode, shape):
    W, H, D, bs = shape
    for minD, swap in ((0, False), (-(D - 1), True), (3, False)):
        for (uq, d12, sw) in [(10, 1, 100), (0, 1000000, 0), (15, 2, 0)]:
            lg, rg = gray_pair(W, H, D, 3 + mode, quant=16 if bs == 5 else 0)
            if swap:
                lg, rg = rg, lg
            kw = dict(minDisparity=minD, numDisparities=D, blockSize=bs, P1=24 * bs * bs, P2=96 * bs * bs,
                      disp12MaxDiff=d12, preFilterCap=63, uniquenessRatio=uq, speckleWindowSize=sw, speckleRange=32,
                      mode=mode)
            tag = "m%d %s minD%d u%d" % (mode, shape, minD, uq)
            want = cv2.StereoSGBM_create(**kw).compute(lg, rg)
            p = N.SgbmParams(**kw)
            if mode != 2:
                disp, raw, Cg, Sg = ctx.sgbm_compute(p, lg, rg, want_raw=True, want_volumes=True)
                _, oraw, oC, oS = cref.sgbm_compute(lg, rg, want_volumes=True, want_raw=True, **kw)
                eq(Cg, oC, tag + " C volume")
                eq(Sg, oS, tag + " S volume")
            else:
                disp, raw = ctx.sgbm_compute(p, lg, rg, want_raw=True)
                _, oraw = cref.sgbm_compute(lg, rg, want_raw=True, **kw)
            eq(raw, oraw, tag + " raw")
            eq(disp, want, tag + " disp vs cv2")
            # production path (WTA fused into the last aggregation path, no S volume written)
            eq(ctx.sgbm_compute(p, lg, rg), want, tag + " fused-WTA disp vs cv2")


# the matcher pair of get_frames() in one call: one pixel-cost pass feeds both cost volumes (sgbm_cost_dual_kernel);
# widths chosen so that the sheared range [RA, RB) is empty, a few columns, and most of the volume
PAIR_SHAPES = [(200, 40, 64, 5), (330, 50, 64, 5), (320, 360, 64, 5), (300, 30, 128, 9), (420, 44, 128, 9),
               (533, 37, 128, 9), (1280, 720, 128, 9), (260, 40, 32, 5), (400, 40, 128, 7), (300, 30, 256, 11),
               (600, 40, 256, 11), (1920, 48, 256, 11)]


@pytest.mark.parametrize("mode", [1, 0, 3, 2])
@pytest.mark.parametrize("shape", PAIR_SHAPES)
def test_sgbm_pair_shared_cost_pass(ctx, mode, shape):
    W, H, D, bs = shape
    if W >= 1280 and mode in (2, 3):
        pytest.skip("full size only in the modes the shared pass serves by default")
    lg, rg = gray_pair(W, H, D, 5, quant=8 if (W == 330 or W == 420) else 0)
    _, mut, right = ref_ops.sgbm_param_sets(D, bs, mode)
    pl, pr = N.SgbmParams(**mut), N.SgbmParams(**right)
    if mode == 2:
        dl, dr = ctx.sgbm_compute_pair(pl, pr, lg, rg)
    else:
        dl, dr, Cl, Cr = ctx.sgbm_compute_pair(pl, pr, lg, rg, want_volumes=True)
        if H <= 64:  # the C restatement of the oracle, cv2 never exposes the volumes
            _, oCl, _ = cref.sgbm_compute(lg, rg, want_volumes=True, **mut)
            _, oCr, _ = cref.sgbm_compute(rg, lg, want_volumes=True, **right)
        else:        # the single-matcher path (itself checked against the oracle above)
            _, oCl, _ = ctx.sgbm_compute(pl, lg, rg, want_volumes=True)
            _, oCr, _ = ctx.sgbm_compute(pr, rg, lg, want_volumes=True)
        eq(Cl, oCl, "%s m%d left cost volume" % (shape, mode))
        eq(Cr, oCr, "%s m%d right cost volume" % (shape, mode))
    eq(dl, cv2.StereoSGBM_create(**mut).compute(lg, rg), "%s m%d left disparity vs cv2" % (shape, mode))
    eq(dr, cv2.StereoSGBM_create(**right).compute(rg, lg), "%s m%d right disparity vs cv2" % (shape, mode))


def test_sgbm_int16_domain_guard(ctx):
    """cv2 keeps the cost volume in int16 and wraps when block sum + P2 reaches 32768; this library carries unsigned 16-bit
    pairs, so beyond that point the bits would differ silently.  The cost kernels flag the event on the device and the
    call fails with L3D_ERR_UNSUPPORTED instead.  With the reference's own penalties (P2 = 96 bs^2) an adversarial
    sawtooth pair at block 11 stays inside the domain (max C = 30976) and must equal cv2."""
    W, H, D = 200, 48, 32
    x = np.arange(W)
    saw = ((x % 32) * 8).astype(np.uint8)
    l, r = np.tile(saw, (H, 1)), np.tile(255 - saw, (H, 1))
    noise = np.random.default_rng(1).integers(0, 256, (H, W), dtype=np.uint8)
    kw = dict(minDisparity=0, numDisparities=D, blockSize=11, P1=2904, P2=11616, disp12MaxDiff=1, preFilterCap=63,
              uniquenessRatio=10, speckleWindowSize=0, speckleRange=0, mode=1)
    eq(ctx.sgbm_compute(N.SgbmParams(**kw), l, r), cv2.StereoSGBM_create(**kw).compute(l, r), "sawtooth, reference penalties")
    for (a, b, bs) in ((l, r, 11), (noise, 255 - noise, 15)):
        bad = dict(kw, blockSize=bs, P1=4000, P2=16000)
        with pytest.raises(N.L3DError, match="int16"):
            ctx.sgbm_compute(N.SgbmParams(**bad), a, b)
        with pytest.raises(N.L3DError, match="int16"):
            ctx.sgbm_compute_pair(N.SgbmParams(**bad), N.SgbmParams(**dict(bad, minDisparity=-(D - 1))), a, b)
    # the context stays usable
    eq(ctx.sgbm_compute(N.SgbmParams(**kw), l, r), cv2.StereoSGBM_create(**kw).compute(l, r), "after the error")


@pytest.mark.parametrize("mode", [2, 0, 1, 3])
def test_sgbm_c1_parameter_sets(ctx, mode):
    lg, rg = gray_pair(320, 360, 64, 7)
    base, mut, right = ref_ops.sgbm_param_sets(64, 5, mode)
    eq(ctx.sgbm_compute(N.SgbmParams(**base), lg, rg), cv2.StereoSGBM_create(**base).compute(lg, rg), "as constructed")
    eq(ctx.sgbm_compute(N.SgbmParams(**mut), lg, rg), cv2.StereoSGBM_create(**mut).compute(lg, rg), "wls-mutated")
    eq(ctx.sgbm_compute(N.SgbmParams(**right), rg, lg), cv2.StereoSGBM_create(**right).compute(rg, lg), "right matcher")


def test_sgbm_real_pairs(ctx, golden_real):
    base, _, _ = ref_ops.sgbm_param_sets(64, 5, 2)
    for tag in ("a", "b"):
        lg = cv2.cvtColor(golden_real["lrect_" + tag], cv2.COLOR_BGR2GRAY)
        rg = cv2.cvtColor(golden_real["rrect_" + tag], cv2.COLOR_BGR2GRAY)
        eq(ctx.sgbm_compute(N.SgbmParams(**base), lg, rg), golden_real["disp16_" + tag], "real pair " + tag)


@pytest.mark.parametrize("mode", [1, 0, 2, 3])
def test_sgbm_c3_full_size(ctx, mode):
    """BASELINE config 3: 1280x720, 128 disparities, block 9."""
    lg, rg = gray_pair(1280, 720, 128, 11)
    base, mut, right = ref_ops.sgbm_param_sets(128, 9, mode)
    eq(ctx.sgbm_compute(N.SgbmParams(**mut), lg, rg), cv2.StereoSGBM_create(**mut).compute(lg, rg), "c3 wls-mutated")
    if mode == 1:
        eq(ctx.sgbm_compute(N.SgbmParams(**right), rg, lg), cv2.StereoSGBM_create(**right).compute(rg, lg), "c3 right")
        eq(ctx.sgbm_compute(N.SgbmParams(**base), lg, rg), cv2.StereoSGBM_create(**base).compute(lg, rg), "c3 base")


def test_sgbm_c4_full_size(ctx):
    """BASELINE config 4: 1920x1080, 256 disparities, block 11, MODE_HH."""
    lg, rg = gray_pair(1920, 1080, 256, 5)
    _, mut, _ = ref_ops.sgbm_param_sets(256, 11, 1)
    eq(ctx.sgbm_compute(N.SgbmParams(**mut), lg, rg), cv2.StereoSGBM_create(**mut).compute(lg, rg), "c4")


def test_c4_full_pipeline(ctx):
    """BASELINE config 4 through the whole frame pipeline at full size (1920x1080, 256 disparities, block 11, MODE_HH,
    matcher pair + WLS + ImprovedSteger + 3D): the grouped pipeline (shared pixel-cost pass on 32-column tiles,
    cluster-fused aggregation with 8 warps x 13 columns per CTA on 16-CTA clusters) must equal the lane-per-frame
    pipeline (direction-split aggregation) bit for bit, the matcher pair must equal cv2, and the frame must pass the
    north_star acceptance list against the reference path."""
    W, H, D, bs, mode = 1920, 1080, 256, 11, 1
    K, Q = synth.camera_model(W, H)
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    frames = [synth.stereo_pair(W, H, D, 70 + s) for s in range(2)]
    idx = [0, 1, 0, 1, 0, 1, 0]  # one full lane set of seven frames
    L = np.stack([frames[i][0] for i in idx])
    R = np.stack([frames[i][1] for i in idx])
    results = {}
    for lanes in (2, 7):
        cfg = pipeline.make_pipeline_config(W, H, D, bs, mode, Q, K, extractor=N.STEGER_IMPROVED, lanes=lanes, max_points=20000)
        fp = pipeline.FramePipeline(cfg, maps=maps, ctx=ctx)
        try:
            n = 2 if lanes == 2 else 7
            dl, dr = fp.upload(L[:n]), fp.upload(R[:n])
            fp.run_dev(dl, dr, n)
            results[lanes] = [fp.fetch(i) for i in (0, 1)] + ([fp.fetch(6)] if lanes == 7 else [])
        finally:
            fp.close()
    for i in (0, 1):
        for k in ("left_rect", "depth", "disp16", "points_2d", "points_3d"):
            eq(results[2][i][k], results[7][i][k], "c4 grouped vs per-lane %s frame %d" % (k, i))
    eq(results[7][2]["disp16"], results[7][0]["disp16"], "same input in another lane of the set")
    wrect, wdepth, aux = ref_ops.depth_path(frames[1][0], frames[1][1], maps, D, bs, mode, Q, want_all=True)
    got = results[7][1]
    eq(got["left_rect"], wrect, "c4 rectified image vs cv2.remap")
    _, mut, right = ref_ops.sgbm_param_sets(D, bs, mode)
    dl16, dr16 = ctx.sgbm_compute_pair(N.SgbmParams(**mut), N.SgbmParams(**right), aux["lg"], aux["rg"])
    eq(dl16, aux["dl"], "c4 left disparity vs cv2")
    eq(dr16, aux["dr"], "c4 right disparity vs cv2")
    diff = np.abs(got["disp16"].astype(np.int32) - aux["df"].astype(np.int32))
    assert (diff <= 1).mean() >= 0.999
    assert point_sets_agree(got["points_2d"], ref_ops.improved_steger_extract(wrect))


@pytest.mark.parametrize("mode", [0, 1, 2, 3])
def test_sgbm_noise_saturation(ctx, mode):
    rng = np.random.default_rng(0)
    ln = rng.integers(0, 256, (96, 400)).astype(np.uint8)
    rn = rng.integers(0, 256, (96, 400)).astype(np.uint8)
    kw = dict(minDisparity=0, numDisparities=256, blockSize=11, P1=2904, P2=11616, disp12MaxDiff=1000000,
              preFilterCap=63, uniquenessRatio=0, speckleWindowSize=0, speckleRange=32, mode=mode)
    eq(ctx.sgbm_compute(N.SgbmParams(**kw), ln, rn), cv2.StereoSGBM_create(**kw).compute(ln, rn))


def test_sgbm_properties_full_size(ctx):
    """Size-independent properties at c3: determinism, invalid border columns, and shift
    equivariance (a frame made of two different halves stacked vertically far apart matches the
    halves' own results away from the seam for the row-local 3WAY mode's horizontal structure)."""
    lg, rg = gray_pair(1280, 720, 128, 3)
    _, mut, _ = ref_ops.sgbm_param_sets(128, 9, 1)
    p = N.SgbmParams(**mut)
    a = ctx.sgbm_compute(p, lg, rg)
    b = ctx.sgbm_compute(p, lg, rg)
    eq(a, b, "determinism")
    assert np.all(a[:, :128 - 1] == -16)  # columns < minX1 (minus the 3x3 median reach) invalid
    valid = a[:, 140:] >= 0
    assert valid.mean() > 0.9
    # right(x) = left(x + d(x)): the disparity seen at left pixel x is d evaluated at the matching right pixel
    field = np.rint(synth.disparity_field(1280, 720, 128))
    xs = np.arange(1280)[None, :] - np.rint(a / 16.0).astype(np.int64)
    truth = np.take_along_axis(field, np.clip(xs, 0, 1279), axis=1)[:, 140:]
    err = np.abs(a[:, 140:] / 16.0 - truth)[valid]
    assert np.median(err) < 0.6  # the matcher recovers the rendered disparity field


@pytest.mark.parametrize("bs,H", [(11, 8), (11, 20), (11, 24), (11, 28), (9, 20), (5, 12), (3, 8), (9, 5)])
def test_sgbm_3way_tiny_images(ctx, bs, H):
    """SGBM_3WAY on images of a few rows: OpenCV's shifted stripe rows (tests/test_oracle_cv2.py has the story) on the GPU,
    through that mode's stand-alone winner-takes-all, with and without the raw disparity read back."""
    for D, W, seed in ((48, 194, 5), (16, 90, 9)):
        lg, rg = gray_pair(W, H, D, seed)
        for (uq, d12, sw) in ((0, 5, 200), (10, 1, 0)):
            kw = dict(minDisparity=0, numDisparities=D, blockSize=bs, P1=100, P2=1000, disp12MaxDiff=d12, preFilterCap=63,
                      uniquenessRatio=uq, speckleWindowSize=sw, speckleRange=2, mode=2)
            want = cv2.StereoSGBM_create(**kw).compute(lg, rg)
            p = N.SgbmParams(**kw)
            eq(ctx.sgbm_compute(p, lg, rg), want, "3way tiny %s" % ((bs, H, D, uq),))
            disp, raw = ctx.sgbm_compute(p, lg, rg, want_raw=True)
            eq(disp, want, "3way tiny (raw read back) %s" % ((bs, H, D, uq),))


def stripes_3way(H, bs):
    """OpenCV's SGBM_3WAY stripes (make_geom): 4 stripes of ceil(H / 4) rows, each starting `overlap` rows early, clamped
    at row 0.  -> [(first image row, rows)] in volume-row order."""
    stripe = -(-H // 4)
    overlap = bs // 2 + 1 + math.ceil(0.1 * stripe)
    out = []
    for s in range(4):
        y0, y1 = max(s * stripe - overlap, 0), min((s + 1) * stripe, H)
        if y1 > y0:
            out.append((y0, y1 - y0))
    return out


@pytest.mark.parametrize("H", [5, 12, 20, 28, 300])
@pytest.mark.parametrize("bs,D", [(5, 64), (9, 128), (11, 256)])
def test_sgbm_3way_striped_volumes(ctx, bs, D, H):
    """SGBM_3WAY at the (blockSize, numDisparities) pairs the cost kernels are specialised for, from images of a few rows
    (shifted stripe rows) to a few hundred, three or more column tiles wide, in both matcher roles.  The striped cost
    volume must equal the full-image volume of the oracle wherever a stripe's vertical window is not cut at its top:
    every row of a stripe that starts at image row 0, and rows y >= y0 + bs // 2 of the others."""
    W = D + 150
    lg, rg = gray_pair(W, H, D, 13)
    _, mut, right = ref_ops.sgbm_param_sets(D, bs, 2)
    vols = []
    for kw, a, b in ((mut, lg, rg), (right, rg, lg)):
        tag = "3way bs%d D%d H%d minD%d" % (bs, D, H, kw["minDisparity"])
        p = N.SgbmParams(**kw)
        disp, raw, Cg, _ = ctx.sgbm_compute(p, a, b, want_raw=True, want_volumes=True)
        eq(disp, cv2.StereoSGBM_create(**kw).compute(a, b), tag + " disp vs cv2")
        eq(raw, cref.sgbm_compute(a, b, want_raw=True, **kw)[1], tag + " raw")
        _, oC, _ = cref.sgbm_compute(a, b, want_volumes=True, **dict(kw, mode=1))
        vr0 = 0
        for y0, rows in stripes_3way(H, bs):
            first = 0 if y0 == 0 else min(bs // 2, rows)
            eq(Cg[vr0 + first:vr0 + rows], oC[y0 + first:y0 + rows], tag + " C volume, stripe from row %d" % y0)
            vr0 += rows
        assert vr0 == len(Cg), tag + " volume rows"
        vols.append(Cg)
    _, _, Cl, Cr = ctx.sgbm_compute_pair(N.SgbmParams(**mut), N.SgbmParams(**right), lg, rg, want_volumes=True)
    eq(Cl, vols[0], "3way bs%d D%d H%d pair: left volume" % (bs, D, H))
    eq(Cr, vols[1], "3way bs%d D%d H%d pair: right volume" % (bs, D, H))


@pytest.mark.parametrize("H", [1, 2, 3, 5, 8])
def test_sgbm_hh4_short_images(ctx, H):
    """MODE_HH4's constant bottom rows of C (oracle/csrc/orc_sgbm.c) on images shorter than the window."""
    lg, rg = gray_pair(160, H, 32, 11)
    for bs in (3, 7, 11):
        kw = dict(minDisparity=0, numDisparities=32, blockSize=bs, P1=24 * bs * bs, P2=96 * bs * bs, disp12MaxDiff=1,
                  preFilterCap=63, uniquenessRatio=10, speckleWindowSize=0, speckleRange=32, mode=3)
        eq(ctx.sgbm_compute(N.SgbmParams(**kw), lg, rg), cv2.StereoSGBM_create(**kw).compute(lg, rg), "hh4 H=%d bs=%d" % (H, bs))


def test_pipeline_mode_hh4(ctx):
    """The frame pipeline with MODE_HH4 matchers (direction-split aggregation even with many lanes) against the oracle path."""
    W, H, D, bs = 320, 120, 64, 5
    K, Q = synth.camera_model(W, H)
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    frames = [synth.stereo_pair(W, H, D, 70 + s) for s in range(3)]
    L = np.stack([f[0] for f in frames]); R = np.stack([f[1] for f in frames])
    cfg = pipeline.make_pipeline_config(W, H, D, bs, 3, Q, K, extractor=N.STEGER_IMPROVED, lanes=14, max_points=8000)
    fp = pipeline.FramePipeline(cfg, maps=maps, ctx=ctx)
    try:
        fp.run_dev(fp.upload(L), fp.upload(R), len(frames))
        got = fp.fetch(2)
    finally:
        fp.close()
    wrect, wdepth, aux = ref_ops.depth_path(frames[2][0], frames[2][1], maps, D, bs, 3, Q, want_all=True)
    eq(got["left_rect"], wrect, "hh4 pipeline rectified image")
    diff = np.abs(got["disp16"].astype(np.int32) - aux["df"].astype(np.int32))
    assert (diff <= 1).mean() >= 0.999


def test_init_undistort_rectify_map_vs_cv2(ctx, rect_cases):
    """SURVEY 8f N3: cv2.initUndistortRectifyMap on the GPU, bit-exact f32 maps (real rig at two sizes, a synthetic rig
    with 12 distortion coefficients at 1280x720), and the rectified image that follows from them."""
    for K, d, R, P, size in rect_cases:
        mx, my = cv2.initUndistortRectifyMap(K, d, R, P, size, cv2.CV_32FC1)
        gx, gy = ctx.init_undistort_rectify_map(K, d, R, P, size)
        eq(gx, mx, "mapx %s" % (size,))
        eq(gy, my, "mapy %s" % (size,))
    with pytest.raises(N.L3DError):
        ctx.init_undistort_rectify_map(K, np.r_[d, 0.01, 0.0], R, P, size)  # tilted sensor model


BM_CASES = [(320, 121, 64, 15), (200, 60, 32, 9), (400, 90, 128, 21), (160, 40, 16, 5), (640, 48, 128, 15), (100, 9, 16, 7),
            (64, 30, 48, 11), (330, 64, 256, 9), (320, 360, 64, 15), (1280, 720, 128, 15)]


@pytest.mark.parametrize("case", BM_CASES)
def test_stereobm_vs_cv2(ctx, case):
    """cv2.StereoBM (readme.md:392-397, SURVEY 8f N4) on the GPU, bit-exact against the cv2 binary."""
    W, H, D, bs = case
    lg, rg = gray_pair(W, H, D, 21)
    if W == 160:  # heavy ties
        lg, rg = (lg // 32 * 32).astype(np.uint8), (rg // 32 * 32).astype(np.uint8)
    big = W * H > 200000
    d12_ok = bs <= 21
    for minD in ((0,) if big else (0, -8, -(D - 1))):
        for cap, tex, uq, sw, sr, d12 in (((31, 10, 15, 0, 0, -1), (63, 0, 0, 100, 32, -1), (31, 0, 0, 100, 32, 1)) if big else
                                         ((31, 10, 15, 0, 0, -1), (63, 0, 0, 100, 32, -1), (31, 0, 0, 100, 32, 1), (15, 50, 5, 50, 2, 0), (1, 10, 15, 0, 0, 5))):
            if d12 >= 0 and (cap > 31 or not d12_ok):
                continue
            m = cv2.StereoBM_create(numDisparities=D, blockSize=bs)
            m.setMinDisparity(minD); m.setPreFilterCap(cap); m.setTextureThreshold(tex); m.setUniquenessRatio(uq)
            m.setSpeckleWindowSize(sw); m.setSpeckleRange(sr); m.setDisp12MaxDiff(d12)
            got = ctx.bm_compute(N.BmParams(minD, D, bs, cap, tex, uq, sw, sr, d12), lg, rg)
            eq(got, m.compute(lg, rg), "StereoBM %s minD %d cap %d tex %d uq %d speckle %d/%d d12 %d" % (case, minD, cap, tex, uq, sw, sr, d12))


def test_stereobm_class_and_limits(ctx):
    from laser_3d_reconstruction_b200 import stereo
    lg, rg = gray_pair(320, 120, 64, 5)
    m = stereo.StereoBM_create(numDisparities=64, blockSize=15)
    assert m.getPreFilterCap() == 31 and m.getTextureThreshold() == 10 and m.getUniquenessRatio() == 15
    eq(m.compute(lg, rg), cv2.StereoBM_create(numDisparities=64, blockSize=15).compute(lg, rg), "StereoBM class defaults")
    m.setMinDisparity(3)
    with pytest.raises(N.L3DError):
        m.compute(lg, rg)  # positive minDisparity: OpenCV itself writes past the row end there; unsupported


def test_sgbm_rejects_unsupported(ctx):
    lg, rg = gray_pair(96, 48, 16, 0)
    with pytest.raises(N.L3DError):
        ctx.sgbm_compute(N.SgbmParams(0, 24, 3, 72, 288, 1, 63, 10, 0, 0, 0), lg, rg)  # numDisparities % 16
    with pytest.raises(N.L3DError):
        ctx.sgbm_compute(N.SgbmParams(0, 16, 4, 72, 288, 1, 63, 10, 0, 0, 0), lg, rg)  # even block
    with pytest.raises(ValueError):
        ctx.sgbm_compute(N.SgbmParams(0, 16, 3, 72, 288, 1, 63, 10, 0, 0, 0), lg, rg[:, :-1])


def test_median_speckles(ctx):
    rng = np.random.default_rng(1)
    for t in range(5):
        H, W = (37, 61) if t < 2 else ((360, 320) if t < 4 else (720, 1280))
        d = (rng.integers(-1, 40, (H, W)) * 16 + rng.integers(0, 16, (H, W))).astype(np.int16)
        d[rng.random((H, W)) < 0.3] = -16
        eq(ctx.median3_s16(d), cv2.medianBlur(d, 3), "median")
        e = d.copy()
        cv2.filterSpeckles(e, -16, 25, 32)
        eq(ctx.filter_speckles(d, -16, 25, 32), e, "speckles")
    # large smooth regions (components far bigger than maxSize) and a tiny island
    d = np.full((200, 300), 160, np.int16)
    d[50:53, 60:64] = 1600
    e = d.copy()
    cv2.filterSpeckles(e, -16, 100, 32)
    eq(ctx.filter_speckles(d, -16, 100, 32), e, "island")


# ---- K3 WLS (PARITY UNPINNED: oracle restatement only) + K5a depth ---------------------------
@pytest.mark.parametrize("cfg", [(320, 360, 64, 5, 2), (1280, 720, 128, 9, 1)])
def test_wls_and_depth(ctx, cfg):
    W, H, D, bs, mode = cfg
    lg, rg = gray_pair(W, H, D, 9)
    base, mut, right = ref_ops.sgbm_param_sets(D, bs, mode)
    dl = cv2.StereoSGBM_create(**mut).compute(lg, rg)
    dr = cv2.StereoSGBM_create(**right).compute(rg, lg)
    r = int(np.ceil(0.5 * bs))
    want, wconf = cref.wls_filter(dl, dr, lg, 0, D, r, 8000.0, 1.5, want_conf=True)
    # default solver = partitioned parallel tridiagonal solves.  Tolerance (north_star): <= 1 LSB of the int16 output on
    # >= 99.9 % of the pixels; the confidence map does not depend on the solver
    got, conf = ctx.wls_filter(N.WlsParams(8000.0, 1.5, 0, D, r, 24), dl, dr, lg, want_conf=True)
    diff = np.abs(got.astype(np.int32) - want.astype(np.int32))
    assert (diff <= 1).mean() >= 0.999, "wls: %.5f within 1 LSB, max %d" % ((diff <= 1).mean(), diff.max())
    assert (diff == 0).mean() >= 0.99, "wls: only %.5f of the pixels identical" % (diff == 0).mean()
    assert np.array_equal(conf, wconf)
    # serial solver: the oracle's f32 operation order, bit-identical
    got1 = ctx.wls_filter(N.WlsParams(8000.0, 1.5, 0, D, r, 24, N.WLS_SOLVER_SERIAL), dl, dr, lg)
    assert np.array_equal(got1, want)
    Q = synth.camera_model(W, H)[1]
    eq(ctx.disp_to_depth(want, Q), ref_ops.depth_from_disparity(want, Q), "depth with Q")
    eq(ctx.disp_to_depth(want, None), ref_ops.depth_from_disparity(want, None), "depth default branch")


@pytest.mark.parametrize("W,H,D", [(150, 37, 16), (97, 11, 32), (49, 3, 16), (200, 64, 64)])
def test_wls_ragged_sizes_bit_identical(ctx, W, H, D):
    """FGS solver edge cases: ROI widths that are not a multiple of the 32-column tile, fewer rows/columns than a warp's
    ten lines, single-tile rows.  The GPU repeats the oracle's f32 operation order, so the output is bit-identical."""
    rng = np.random.default_rng(W * 1000 + H)
    guide = cv2.GaussianBlur(rng.integers(0, 256, (H, W), dtype=np.uint8), (0, 0), 1.2)
    dl = (rng.integers(0, D * 16, (H, W))).astype(np.int16)
    dl[rng.random((H, W)) < 0.1] = -16
    dr = (-rng.integers(0, D * 16, (H, W))).astype(np.int16)
    want, wconf = cref.wls_filter(dl, dr, guide, 0, D, 3, 8000.0, 1.5, want_conf=True)
    got, conf = ctx.wls_filter(N.WlsParams(8000.0, 1.5, 0, D, 3, 24, N.WLS_SOLVER_SERIAL), dl, dr, guide, want_conf=True)
    assert np.array_equal(got, want), "wls ragged: %d pixels differ" % int((got != want).sum())
    assert np.array_equal(conf, wconf)
    # the parallel solver on the same edge cases (chunks of 2-3 elements, lanes without a chunk, a one-element last chunk)
    gotp = ctx.wls_filter(N.WlsParams(8000.0, 1.5, 0, D, 3, 24), dl, dr, guide)
    diff = np.abs(gotp.astype(np.int32) - want.astype(np.int32))
    assert diff.max() <= 1 and (diff == 0).mean() >= 0.99, "parallel solver: max %d, %.4f identical" % (diff.max(), (diff == 0).mean())


@pytest.mark.parametrize("variant", [1, 2, 4, 8, 15])
def test_wls_unpinned_points_are_switchable(ctx, variant):
    """The readings of opencv_contrib's DisparityWLSFilter that no installed binary can pin here (SURVEY A7) are
    parameters of both the oracle and the GPU path; every setting is bit-identical between the two (serial solver), so
    pinning against a real cv2.ximgproc later is a flag flip."""
    from test_oracle_cv2 import wls_case
    W, H, D = 210, 41, 48
    dl, dr, guide = wls_case(W, H, D, 7)
    want, wconf = cref.wls_filter(dl, dr, guide, 0, D, 3, 8000.0, 1.5, want_conf=True, variant=variant)
    base, bconf = cref.wls_filter(dl, dr, guide, 0, D, 3, 8000.0, 1.5, want_conf=True)
    assert not (np.array_equal(want, base) and np.array_equal(wconf, bconf)), "the variant should change the result on this input"
    got, conf = ctx.wls_filter(N.WlsParams(8000.0, 1.5, 0, D, 3, 24, N.WLS_SOLVER_SERIAL, variant), dl, dr, guide, want_conf=True)
    assert np.array_equal(got, want) and np.array_equal(conf, wconf)


# ---- K4 extractors -------------------------------------------------------------------------
CFG = dict(hsv_lower=(50, 100, 180), hsv_upper=(70, 255, 255), brightness_threshold=200, min_area=50)


def steger_params(variant, sigma=None, roi=(0, 0, 0, 0)):
    return N.StegerParams(variant, (2.0 if variant == 3 else 3.0) if sigma is None else sigma, 200, 0.5,
                          (C.c_int * 4)(*roi), (C.c_int * 3)(50, 100, 180), (C.c_int * 3)(70, 255, 255))


def point_sets_agree(got, want, tol=0.01, frac=0.999):
    got, want = np.asarray(got, np.float64).reshape(-1, 2), np.asarray(want, np.float64).reshape(-1, 2)
    if len(want) == 0 or len(got) == 0:
        return len(want) == len(got)
    from scipy.spatial import cKDTree
    d1 = cKDTree(want).query(got)[0]
    d2 = cKDTree(got).query(want)[0]
    return (d1 <= tol).mean() >= frac and (d2 <= tol).mean() >= frac


@pytest.mark.parametrize("size", [(320, 360, 64), (1280, 720, 128)])
def test_simple_extractor(ctx, size):
    W, H, D = size
    left, _ = synth.stereo_pair(W, H, D, 1)
    wpts, wm1, wm2 = ref_ops.simple_extract(left, want_masks=True, **CFG)
    pts, m1, m2 = ctx.simple_extract(left, CFG["hsv_lower"], CFG["hsv_upper"], 200, 50, want_masks=True)
    eq(m1, wm1, "mask after morphology")
    eq(m2, wm2, "final contour mask")
    eq(pts, np.array(wpts).reshape(-1, 2), "centroids")  # exact: integer sums, one f64 divide
    assert len(pts) == H


def test_simple_extractor_blobs(ctx):
    rng = np.random.default_rng(5)
    for t in range(12):
        m = (cv2.GaussianBlur(rng.random((90, 120)).astype(np.float32), (0, 0), 1.5 + 0.15 * t) > 0.5)
        img = np.zeros((90, 120, 3), np.uint8)
        img[m] = (140, 255, 140)
        wpts, wm1, wm2 = ref_ops.simple_extract(img, want_masks=True, **dict(CFG, min_area=8 + t))
        pts, m1, m2 = ctx.simple_extract(img, CFG["hsv_lower"], CFG["hsv_upper"], 200, 8 + t, want_masks=True)
        eq(m1, wm1, "blob morph %d" % t)
        eq(m2, wm2, "blob final %d" % t)
        eq(pts, np.array(wpts, np.float64).reshape(-1, 2), "blob points %d" % t)


@pytest.mark.parametrize("size", [(320, 360, 64), (1280, 720, 128)])
def test_steger_variants(ctx, size):
    W, H, D = size
    left, _ = synth.stereo_pair(W, H, D, 1)
    for variant, fn in ((0, ref_ops.fast_steger_extract), (1, ref_ops.improved_steger_extract),
                        (2, ref_ops.improved_steger_extract_optimized), (3, ref_ops.hybrid_extract)):
        got = ctx.steger_extract(steger_params(variant), left)
        want = np.array(fn(left), np.float64).reshape(-1, 2)
        assert len(want) > 100
        assert point_sets_agree(got, want), "variant %d: %d vs %d points" % (variant, len(got), len(want))
        if got.shape == want.shape:  # raster order preserved -> element-wise tolerance 0.01 px
            assert np.abs(got - want).max() <= 0.01


def test_extractors_on_golden(ctx, golden_synth):
    """Against outputs of the REAL reference classes (tests/golden/make_golden.py)."""
    g = golden_synth
    left = g["left"]
    eq(ctx.simple_extract(left, CFG["hsv_lower"], CFG["hsv_upper"], 200, 50), g["simple_cfg"], "simple cfg")
    eq(ctx.simple_extract(left, (40, 50, 100), (80, 255, 255), 100, 50), g["simple_def"], "simple defaults")
    for variant, key in ((0, "fast"), (1, "improved"), (2, "optimized"), (3, "hybrid")):
        got = ctx.steger_extract(steger_params(variant), left)
        assert got.shape == g[key].shape and np.abs(got - g[key]).max() <= 0.01, key
    got = ctx.steger_extract(steger_params(0, roi=(100, 40, 150, 200)), left)
    assert got.shape == g["fast_roi"].shape and np.abs(got - g["fast_roi"]).max() <= 0.01
    gray = cv2.cvtColor(left, cv2.COLOR_BGR2GRAY)
    got = ctx.steger_extract(steger_params(0), gray)
    assert got.shape == g["fast_gray"].shape and np.abs(got - g["fast_gray"]).max() <= 0.01


def test_extractors_empty_image(ctx):
    dark = np.full((64, 96, 3), 40, np.uint8)
    assert len(ctx.simple_extract(dark, CFG["hsv_lower"], CFG["hsv_upper"], 200, 50)) == 0
    for v in range(4):
        assert len(ctx.steger_extract(steger_params(v), dark)) == 0


# ---- K5b reconstruction ----------------------------------------------------------------------
def test_reconstruction_on_golden(ctx, golden_synth):
    g = golden_synth
    K, Q = g["K"], g["Q"]
    sp = g["simple_cfg"]

    def rp(kind, refr=0):
        p = N.ReconParams()
        p.kind = kind
        p.K[:] = list(K.reshape(9))
        p.plane[:] = list(synth.LASER_PLANE)
        p.use_refraction = refr
        p.n_water = 1.33
        return p

    for name, refr in (("rec_air", 0), ("rec_water", 1)):
        got = ctx.reconstruct(rp(N.RECON_PLANE, refr), sp)
        want = g[name + "_line"]
        assert got.shape == want.shape and np.allclose(got, want, rtol=1e-9, atol=1e-12), name  # north_star: <= 1e-5 rel
        eq(ctx.reconstruct(rp(N.RECON_DEPTH), sp, g["depth"]), g[name + "_depth"], name + " depth")
    got = ctx.reconstruct(rp(N.RECON_DEPTH), g["fast"].astype(np.float64), g["depth"])
    eq(got, g["rec_fast_depth"], "from_depth with float32 points")
    disp = g["disp16_3way"].astype(np.float32) / 16.0
    ir = ref_ops.ImprovedLaserReconstructorRef(Q)
    for kind, key in ((N.RECON_DISPARITY, "irec_disp"), (N.RECON_DISPARITY_MEDIAN, "irec_interp")):
        p = N.ReconParams()
        p.kind = kind
        p.fx, p.baseline, p.cx, p.cy = ir.fx, ir.baseline, ir.cx, ir.cy
        p.min_disparity = 1.0
        p.window = 3
        eq(ctx.reconstruct(p, g["optimized"], disp).astype(np.float32), g[key], key)
    assert ctx.reconstruct(rp(N.RECON_PLANE), np.zeros((0, 2))).shape == (0, 3)


# ---- fused depth path + frame pipeline ---------------------------------------------------------
@pytest.mark.parametrize("cfg", [(320, 360, 64, 5, 2, True), (320, 360, 64, 5, 0, False), (1280, 720, 128, 9, 1, True)])
def test_compute_depth_fused(ctx, cfg):
    W, H, D, bs, mode, use_wls = cfg
    left, right = synth.stereo_pair(W, H, D, 4)
    K, Q = synth.camera_model(W, H)
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    ctx.set_rectify_maps(0, maps[0], maps[1])
    ctx.set_rectify_maps(1, maps[2], maps[3])
    dc = pipeline.depth_config(D, bs, mode, Q, use_wls=use_wls)
    rect, depth, disp = ctx.compute_depth(dc, left, right, want_disp=True)
    wrect, wdepth, aux = ref_ops.depth_path(left, right, maps, D, bs, mode, Q, use_wls=use_wls, want_all=True)
    eq(rect, wrect, "rectified left")
    if use_wls:
        diff = np.abs(disp.astype(np.int32) - aux["df"].astype(np.int32))
        assert (diff <= 1).mean() >= 0.999
        ok = diff == 0
        assert np.array_equal(depth[ok], wdepth[ok])
    else:
        eq(disp, aux["df"], "disparity")
        eq(depth, wdepth, "depth")


def test_pipeline_matches_stagewise_and_is_frame_independent(ctx):
    W, H, D, bs = 320, 360, 64, 5
    K, Q = synth.camera_model(W, H)
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    frames = [synth.stereo_pair(W, H, D, s) for s in range(5)]
    L = np.stack([f[0] for f in frames])
    R = np.stack([f[1] for f in frames])
    results = {}
    for lanes in (1, 3):
        cfg = pipeline.make_pipeline_config(W, H, D, bs, 2, Q, K, extractor=N.STEGER_IMPROVED, lanes=lanes, max_points=8000)
        fp = pipeline.FramePipeline(cfg, maps=maps, ctx=ctx)
        try:
            dl, dr = fp.upload(L), fp.upload(R)
            counts = fp.run_dev(dl, dr, len(frames))
            results[lanes] = [fp.fetch(i) for i in range(len(frames))]
            assert list(counts) == [len(r["points_3d"]) for r in results[lanes]]
            # device-side packing of the point clouds (payload of the NCCL gather to rank 0)
            ids = [100 + 7 * i for i in range(len(frames))]
            nrows = int(np.sum(counts))
            buf = ctx.lib.l3d_dev_alloc(ctx.h, max(nrows, 1) * 32)
            assert fp.pack_points_dev(ids, buf) == nrows
            table = np.empty((nrows, 4), np.float64)
            ctx.check(ctx.lib.l3d_memcpy_d2h(ctx.h, table.ctypes.data, buf, table.nbytes), "d2h")
            ctx.lib.l3d_dev_free(ctx.h, buf)
            from laser_3d_reconstruction_b200 import sharding
            back = sharding.unpack_clouds(np.concatenate([table[:, :1] - 100, table[:, 1:]], axis=1) / [7, 1, 1, 1], len(frames))
            for i in range(len(frames)):
                eq(back[i], results[lanes][i]["points_3d"], "packed points frame %d" % i)
            # host-buffer entry point gives the same answer
            depth = np.empty((len(frames), H, W), np.float32)
            xyz = np.empty((len(frames), 8000, 3), np.float64)
            counts2 = fp.run_host(L, R, depth, xyz)
            assert list(counts2) == list(counts)
            for i in range(len(frames)):
                eq(depth[i], results[lanes][i]["depth"], "run_host depth")
                eq(xyz[i, :counts[i]], results[lanes][i]["points_3d"], "run_host xyz")
        finally:
            fp.close()
    for i in range(len(frames)):  # lanes (streams) do not change any bit
        for k in ("left_rect", "depth", "disp16", "points_2d", "points_3d"):
            eq(results[1][i][k], results[3][i][k], "lanes %s frame %d" % (k, i))
    # frame 2 against the stage-wise reference path
    wrect, wdepth, aux = ref_ops.depth_path(frames[2][0], frames[2][1], maps, D, bs, 2, Q, want_all=True)
    got = results[1][2]
    eq(got["left_rect"], wrect, "pipeline rect")
    diff = np.abs(got["disp16"].astype(np.int32) - aux["df"].astype(np.int32))
    assert (diff <= 1).mean() >= 0.999
    wp = ref_ops.improved_steger_extract(wrect)
    assert point_sets_agree(got["points_2d"], wp)
    wxyz = ref_ops.ReconstructorRef(K, synth.LASER_PLANE, False).reconstruct_from_depth(
        [tuple(p) for p in got["points_2d"].astype(np.float64)], got["depth"]).reshape(-1, 3)
    assert got["points_3d"].shape == wxyz.shape
    assert np.allclose(got["points_3d"], wxyz, rtol=1e-5, atol=1e-12)  # north_star: 3D points <= 1e-5 relative


@pytest.mark.parametrize("mode", [1, 0])
def test_grouped_pipeline_cluster_aggregation(ctx, mode):
    """lanes >= 7 switches the frame pipeline to grouped mode: SGBM fronts per lane, ONE cluster-fused
    aggregation launch per pass over all volumes of a lane set (sgbm_vgroup.cu), backs per lane.  Every bit
    must equal the lane-per-frame pipeline (direction-split scan kernels) and cv2."""
    W, H, D, bs = 320, 360, 64, 5
    K, Q = synth.camera_model(W, H)
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    frames = [synth.stereo_pair(W, H, D, 10 + s) for s in range(9)]  # 9 frames: one full lane set of 7 + a ragged one
    L = np.stack([f[0] for f in frames])
    R = np.stack([f[1] for f in frames])
    results = {}
    for lanes in (2, 14):
        cfg = pipeline.make_pipeline_config(W, H, D, bs, mode, Q, K, extractor=N.STEGER_IMPROVED, lanes=lanes, max_points=8000)
        fp = pipeline.FramePipeline(cfg, maps=maps, ctx=ctx)
        try:
            dl, dr = fp.upload(L), fp.upload(R)
            for _ in range(5):  # steady state: scratch reuse across runs; a launch-bound step (this size is) is captured
                fp.run_dev(dl, dr, len(frames))  # on its third occurrence and replayed as a CUDA graph afterwards
            if lanes == 14:
                assert fp.graph_replays >= 1, "the repeated 320x360 step should have been replayed as a CUDA graph"
            results[lanes] = [fp.fetch(i) for i in range(len(frames))]
        finally:
            fp.close()
    for i in range(len(frames)):
        for k in ("left_rect", "depth", "disp16", "points_2d", "points_3d"):
            eq(results[2][i][k], results[14][i][k], "grouped vs per-lane %s frame %d" % (k, i))
    # and the two matcher runs feeding WLS equal cv2 on one frame
    wrect, wdepth, aux = ref_ops.depth_path(frames[8][0], frames[8][1], maps, D, bs, mode, Q, want_all=True)
    diff = np.abs(results[14][8]["disp16"].astype(np.int32) - aux["df"].astype(np.int32))
    assert (diff <= 1).mean() >= 0.999


def test_pipeline_graph_replay_host_buffers(ctx):
    """A repeated launch-bound step through HOST buffers (H2D / D2H copies inside the captured graph): replays give the
    same depth maps and point clouds as the direct launches of the first occurrences, also after the input CONTENT
    changes in place (same pointers, new frames)."""
    W, H, D, bs = 320, 360, 64, 5
    K, Q = synth.camera_model(W, H)
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    cap = 8000
    cfg = pipeline.make_pipeline_config(W, H, D, bs, 1, Q, K, extractor=N.STEGER_IMPROVED, lanes=14, max_points=cap)
    fp = pipeline.FramePipeline(cfg, maps=maps, ctx=ctx)
    try:
        frames = [synth.stereo_pair(W, H, D, 90 + s) for s in range(14)]
        pL = pipeline.pinned_empty((14, H, W, 3), np.uint8); pR = pipeline.pinned_empty((14, H, W, 3), np.uint8)
        depth = pipeline.pinned_empty((14, H, W), np.float32); xyz = pipeline.pinned_empty((14, cap, 3), np.float64)
        pL[:] = np.stack([f[0] for f in frames]); pR[:] = np.stack([f[1] for f in frames])
        counts0 = fp.run_host(pL, pR, depth, xyz)
        d0, x0 = depth.copy(), [xyz[i, :counts0[i]].copy() for i in range(14)]
        for _ in range(4):
            counts = fp.run_host(pL, pR, depth, xyz)
        assert fp.graph_replays >= 1
        assert list(counts) == list(counts0) and np.array_equal(depth, d0)
        for i in range(14):
            assert np.array_equal(xyz[i, :counts[i]], x0[i])
        # new content in the same buffers: the replayed graph must pick it up
        pL[:] = pL[::-1].copy(); pR[:] = pR[::-1].copy()
        counts2 = fp.run_host(pL, pR, depth, xyz)
        assert list(counts2) == list(counts0)[::-1] and np.array_equal(depth, d0[::-1])
    finally:
        fp.close()


@pytest.mark.parametrize("W,H,D,bs", [(1100, 64, 128, 9), (437, 50, 64, 5), (300, 33, 64, 7), (1920, 40, 128, 9), (700, 30, 256, 5),
                                      (1920, 36, 256, 11), (1500, 30, 256, 5),  # these two: 8 warps x 13 / 10 columns, 16-CTA clusters
                                      (1280, 720, 128, 9),  # config 3 at full height: the wavefront kernel's fill, steady state and drain
                                      (640, 5, 128, 5), (700, 3, 128, 5)])  # fewer rows than pipeline stages of the row loop
@pytest.mark.parametrize("policy", [None, "1"])  # L3D_VWAVE: default = the wavefront kernel where it pays, 1 = wherever it applies
def test_grouped_pipeline_ragged_geometry(ctx, W, H, D, bs, policy):
    """Cluster-fused aggregation (MODE_HH at D <= 128: the two-pass wavefront kernel sgbm_vwave.cu, else sgbm_vgroup.cu) on
    volumes that do not fill the cluster's column strips: the last CTA / last warps own fewer (or no) valid columns,
    neighbour-CTA hand-off (st.async + mbarrier) still has to deliver "no predecessor" there.  Grouped (14 lanes) == lane-per-frame (2 lanes, direction-split kernels) bit for bit, and the raw matcher
    output equals cv2."""
    import os
    mode = 1
    if policy is not None and (D > 128 or (W, H) == (1280, 720)):
        pytest.skip("the wavefront kernel does not cover D = 256; config 3 takes it by default")
    K, Q = synth.camera_model(W, H)
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    frames = [synth.stereo_pair(W, H, D, 40 + s) for s in range(8)]
    L = np.stack([f[0] for f in frames])
    R = np.stack([f[1] for f in frames])
    results = {}
    saved = os.environ.get("L3D_VWAVE")
    if policy is not None:
        os.environ["L3D_VWAVE"] = policy  # read by the library when a pipeline is created
    try:
        for lanes in (2, 14):
            cfg = pipeline.make_pipeline_config(W, H, D, bs, mode, Q, K, extractor=N.STEGER_IMPROVED, lanes=lanes, max_points=8000)
            fp = pipeline.FramePipeline(cfg, maps=maps, ctx=ctx)
            try:
                dl, dr = fp.upload(L), fp.upload(R)
                fp.run_dev(dl, dr, len(frames))
                results[lanes] = [fp.fetch(i) for i in range(len(frames))]
            finally:
                fp.close()
    finally:
        if saved is None:
            os.environ.pop("L3D_VWAVE", None)
        else:
            os.environ["L3D_VWAVE"] = saved
    for i in range(len(frames)):
        for k in ("left_rect", "depth", "disp16", "points_2d", "points_3d"):
            eq(results[2][i][k], results[14][i][k], "ragged grouped vs per-lane %s frame %d" % (k, i))
    wrect, wdepth, aux = ref_ops.depth_path(frames[7][0], frames[7][1], maps, D, bs, mode, Q, want_all=True)
    diff = np.abs(results[14][7]["disp16"].astype(np.int32) - aux["df"].astype(np.int32))
    assert (diff <= 1).mean() >= 0.999


def test_grouped_pipeline_is_deterministic(ctx):
    """The same frames through the grouped pipeline (wavefront aggregation: mbarrier hand-offs between skewed warps, relaxed
    remote arrives, st.async slots) twelve times: every output bit equals the first run's.  (tools/stress_determinism.py is
    the long form: config 3 / config 4 sizes, dozens of runs.)"""
    W, H, D, bs = 640, 240, 128, 7
    K, Q = synth.camera_model(W, H)
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    frames = [synth.stereo_pair(W, H, D, 80 + s) for s in range(14)]
    L = np.stack([f[0] for f in frames])
    R = np.stack([f[1] for f in frames])
    cfg = pipeline.make_pipeline_config(W, H, D, bs, 1, Q, K, extractor=N.STEGER_IMPROVED, lanes=14, max_points=8000)
    fp = pipeline.FramePipeline(cfg, maps=maps, ctx=ctx)
    try:
        dl, dr = fp.upload(L), fp.upload(R)
        first = None
        for run in range(12):
            fp.run_dev(dl, dr, len(frames))
            got = [fp.fetch(i) for i in range(len(frames))]
            if first is None:
                first = got
                continue
            for i in range(len(frames)):
                for k in ("disp16", "depth", "points_3d"):
                    eq(first[i][k], got[i][k], "run %d frame %d %s vs run 0" % (run, i, k))
    finally:
        fp.close()


@pytest.mark.parametrize("W,H,D,bs", [(640, 200, 128, 9), (437, 50, 64, 5)])
def test_grouped_pipeline_without_wls_uniqueness(ctx, W, H, D, bs):
    """use_wls = False: one matcher per frame with the reference's own parameters (uniquenessRatio 10, disp12MaxDiff 1,
    speckle filter): the fused winner-takes-all of the cluster kernels (wavefront kernel forced on: L3D_VWAVE=1) runs
    OpenCV's uniqueness test.  Grouped (15 lanes) == lane-per-frame (2 lanes, direction-split kernels + stand-alone WTA)
    bit for bit, and the disparity equals cv2's."""
    import os
    import cv2
    mode = 1
    K, Q = synth.camera_model(W, H)
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    frames = [synth.stereo_pair(W, H, D, 60 + s) for s in range(9)]
    L = np.stack([f[0] for f in frames])
    R = np.stack([f[1] for f in frames])
    results = {}
    saved = os.environ.get("L3D_VWAVE")
    os.environ["L3D_VWAVE"] = "1"
    try:
        for lanes in (2, 15):
            cfg = pipeline.make_pipeline_config(W, H, D, bs, mode, Q, K, extractor=N.STEGER_IMPROVED, lanes=lanes, max_points=8000,
                                                use_wls=False)
            fp = pipeline.FramePipeline(cfg, maps=maps, ctx=ctx)
            try:
                dl, dr = fp.upload(L), fp.upload(R)
                fp.run_dev(dl, dr, len(frames))
                results[lanes] = [fp.fetch(i) for i in range(len(frames))]
            finally:
                fp.close()
    finally:
        if saved is None:
            os.environ.pop("L3D_VWAVE", None)
        else:
            os.environ["L3D_VWAVE"] = saved
    for i in range(len(frames)):
        for k in ("left_rect", "depth", "disp16", "points_2d", "points_3d"):
            eq(results[2][i][k], results[15][i][k], "no-WLS grouped vs per-lane %s frame %d" % (k, i))
    lrect = cv2.remap(frames[8][0], maps[0], maps[1], cv2.INTER_LINEAR)
    rrect = cv2.remap(frames[8][1], maps[2], maps[3], cv2.INTER_LINEAR)
    want = cv2.StereoSGBM_create(minDisparity=0, numDisparities=D, blockSize=bs, P1=24 * bs * bs, P2=96 * bs * bs, disp12MaxDiff=1,
                                 preFilterCap=63, uniquenessRatio=10, speckleWindowSize=100, speckleRange=32, mode=mode).compute(
        cv2.cvtColor(lrect, cv2.COLOR_BGR2GRAY), cv2.cvtColor(rrect, cv2.COLOR_BGR2GRAY))
    eq(results[15][8]["disp16"], want, "no-WLS grouped disparity vs cv2")

