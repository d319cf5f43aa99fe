"""Pin the oracle's C restatement (oracle/csrc) against the installed cv2 binary -- the library the
reference calls on its hot path (SURVEY 8c).  Bit-exact for every integer stage."""
import cv2

import numpy as np
import pytest

from laser_3d_reconstruction_b200 import synth
from oracle import cref, ref_ops


def gray_pair(W, H, D, seed, quant=0):
    l, r = synth.stereo_pair(W, H, D, seed)
    lg, rg = cv2.cvtColor(l, cv2.COLOR_BGR2GRAY), cv2.cvtColor(r, cv2.COLOR_BGR2GRAY)
    if quant:
        lg = (lg // quant * quant).astype(np.uint8)
        rg = (rg // quant * quant).astype(np.uint8)
    return lg, rg


def test_gray_hsv_colour_cube_slice():
    # a dense slice of the 2^24 cube (every 3rd value per channel + the extremes)
    v = np.unique(np.concatenate([np.arange(0, 256, 3), [254, 255]])).astype(np.uint8)
    b, g, r = np.meshgrid(v, v, v, indexing="ij")
    img = np.stack([b, g, r], -1).reshape(len(v), -1, 3)
    assert np.array_equal(cref.bgr2gray(img), cv2.cvtColor(img, cv2.COLOR_BGR2GRAY))
    assert np.array_equal(cref.bgr2hsv(img), cv2.cvtColor(img, cv2.COLOR_BGR2HSV))


@pytest.mark.parametrize("case", range(4))
def test_remap(case):
    rng = np.random.default_rng(case)
    H, W = (53, 97) if case < 2 else (120, 160)
    src = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    mx = (rng.random((H, W)) * (W + 8) - 4).astype(np.float32)
    my = (rng.random((H, W)) * (H + 8) - 4).astype(np.float32)
    if case == 1:  # exact half-way fixed-point roundings
        mx = (np.round(mx * 64) / 64).astype(np.float32)
        my = (np.round(my * 64) / 64).astype(np.float32)
    if case == 3:
        mx, my = synth.warp_maps(W, H, 1)
    assert np.array_equal(cref.remap_bilinear(src, mx, my), cv2.remap(src, mx, my, cv2.INTER_LINEAR))


SGBM_CASES = [
    # (W, H, D, bs, minD-kind, params-kind, quant)
    (96, 48, 16, 3, "zero", "base", 0), (130, 50, 32, 5, "zero", "base", 16), (130, 50, 32, 5, "right", "mut", 16),
    (200, 64, 64, 9, "zero", "mut", 0), (200, 64, 64, 9, "pos", "base", 0), (300, 56, 128, 7, "zero", "base", 0),
    (300, 56, 128, 7, "right", "mut", 0), (400, 48, 256, 11, "zero", "mut", 0), (180, 52, 96, 5, "pos", "base", 8),
]


@pytest.mark.parametrize("mode", [0, 1, 2, 3])  # 3 = MODE_HH4 (SURVEY 8f N4)
@pytest.mark.parametrize("case", SGBM_CASES)
def test_sgbm_vs_cv2(mode, case):
    W, H, D, bs, mk, pk, quant = case
    lg, rg = gray_pair(W, H, D, 3 + mode, quant)
    minD = {"zero": 0, "right": -(D - 1), "pos": 3}[mk]
    if mk == "right":
        lg, rg = rg, lg
    uq, d12, sw = (10, 1, 100) if pk == "base" else (0, 1000000, 0)
    kw = dict(minDisparity=minD, numDisparities=D, blockSize=bs, P1=24 * bs * bs, P2=96 * bs * bs, disp12MaxDiff=d12,
              preFilterCap=63, uniquenessRatio=uq, speckleWindowSize=sw, speckleRange=32, mode=mode)
    want = cv2.StereoSGBM_create(**kw).compute(lg, rg)
    assert np.array_equal(cref.sgbm_compute(lg, rg, **kw), want)


@pytest.mark.parametrize("mode", [0, 1, 2, 3])
def test_sgbm_c1_and_saturation(mode):
    lg, rg = gray_pair(320, 360, 64, 7)
    base, mut, right = ref_ops.sgbm_param_sets(64, 5, mode)
    assert np.array_equal(cref.sgbm_compute(lg, rg, **base), cv2.StereoSGBM_create(**base).compute(lg, rg))
    assert np.array_equal(cref.sgbm_compute(rg, lg, **right), cv2.StereoSGBM_create(**right).compute(rg, lg))
    # pure noise at bs=11: S saturates at 32767 (all-saturated pixels stay invalid, SURVEY A4)
    rng = np.random.default_rng(0)
    ln = rng.integers(0, 256, (64, 400)).astype(np.uint8)
    rn = rng.integers(0, 256, (64, 400)).astype(np.uint8)
    kw = dict(minDisparity=0, numDisparities=256, blockSize=11, P1=2904, P2=11616, disp12MaxDiff=1000000,
              preFilterCap=63, uniquenessRatio=0, speckleWindowSize=0, speckleRange=32, mode=mode)
    assert np.array_equal(cref.sgbm_compute(ln, rn, **kw), cv2.StereoSGBM_create(**kw).compute(ln, rn))


@pytest.mark.parametrize("bs,H", [(11, 8), (11, 20), (11, 24), (11, 28), (9, 20), (7, 16), (5, 12), (3, 8), (5, 7), (9, 5)])
def test_sgbm_3way_tiny_images(bs, H):
    """SGBM_3WAY on images of a few rows: where a stripe's start is clamped at the image top (ceil(H / 4) < blockSize / 2 + 1
    + ceil(0.1 ceil(H / 4))) OpenCV's stripe buffers and its final assembly do not meet and the output rows of that stripe
    are the results of rows further down (found by differential fuzzing: tests/fuzz/fuzz_oracle.py)."""
    for D, W, seed in ((48, 194, 5), (16, 90, 9)):
        lg, rg = gray_pair(W, H, D, seed)
        for (uq, d12, sw) in ((0, 5, 200), (10, 1, 0)):
            kw = dict(minDisparity=0, numDisparities=D, blockSize=bs, P1=100, P2=1000, disp12MaxDiff=d12, preFilterCap=63,
                      uniquenessRatio=uq, speckleWindowSize=sw, speckleRange=2, mode=2)
            assert np.array_equal(cref.sgbm_compute(lg, rg, **kw), cv2.StereoSGBM_create(**kw).compute(lg, rg)), (D, uq)


@pytest.mark.parametrize("H", [1, 2, 3, 5, 8])
def test_sgbm_hh4_short_images(H):
    """MODE_HH4 leaves the last blockSize/2 rows of the cost volume at P2 (no branch for window rows below the image
    in OpenCV's HH4 cost loop): images shorter than the window exercise every clamp of that rule."""
    lg, rg = gray_pair(160, H, 32, 11)
    for bs in (3, 7, 11):
        kw = dict(minDisparity=0, numDisparities=32, blockSize=bs, P1=24 * bs * bs, P2=96 * bs * bs, disp12MaxDiff=1,
                  preFilterCap=63, uniquenessRatio=10, speckleWindowSize=0, speckleRange=32, mode=3)
        assert np.array_equal(cref.sgbm_compute(lg, rg, **kw), cv2.StereoSGBM_create(**kw).compute(lg, rg)), (H, bs)


def test_sgbm_real_pair(golden_real):
    """int16 disparity of the real 320x240 pair as the reference's camera class computed it."""
    g = golden_real
    base, _, _ = ref_ops.sgbm_param_sets(64, 5, 2)
    for tag in ("a", "b"):
        lg = cv2.cvtColor(g["lrect_" + tag], cv2.COLOR_BGR2GRAY)
        rg = cv2.cvtColor(g["rrect_" + tag], cv2.COLOR_BGR2GRAY)
        assert np.array_equal(cref.sgbm_compute(lg, rg, **base), g["disp16_" + tag])


BM_CASES = [(320, 121, 64, 15), (200, 60, 32, 9), (400, 90, 128, 21), (160, 40, 16, 5), (640, 48, 128, 15), (100, 9, 16, 7),
            (64, 30, 48, 11)]


@pytest.mark.parametrize("case", BM_CASES)
def test_stereobm_vs_cv2(case):
    """cv2.StereoBM (readme.md:392-397, SURVEY 8f N4): the restatement against the cv2 binary, bit-exact, over the
    parameters its setters expose (minDisparity <= 0, disp12MaxDiff off)."""
    W, H, D, bs = case
    lg, rg = gray_pair(W, H, D, 21)
    if W == 160:  # heavy ties
        lg, rg = (lg // 32 * 32).astype(np.uint8), (rg // 32 * 32).astype(np.uint8)
    for minD in (0, -8, -(D - 1)):
        for cap, tex, uq, sw, sr, d12 in ((31, 10, 15, 0, 0, -1), (63, 0, 0, 100, 32, -1), (31, 0, 0, 100, 32, 1), (15, 50, 5, 50, 2, 0), (1, 10, 15, 0, 0, 5)):
            m = cv2.StereoBM_create(numDisparities=D, blockSize=bs)
            m.setMinDisparity(minD); m.setPreFilterCap(cap); m.setTextureThreshold(tex); m.setUniquenessRatio(uq)
            m.setSpeckleWindowSize(sw); m.setSpeckleRange(sr); m.setDisp12MaxDiff(d12)
            got = cref.bm_compute(lg, rg, D, bs, minD, cap, tex, uq, sw, sr, d12)
            assert np.array_equal(got, m.compute(lg, rg)), (case, minD, cap, tex, uq, sw, sr, d12)


def test_init_undistort_rectify_map_vs_cv2(rect_cases):
    """SURVEY 8f N3: the f64 restatement of cv2.initUndistortRectifyMap gives cv2's f32 maps bit for bit."""
    for K, d, R, P, size in rect_cases:
        mx, my = cv2.initUndistortRectifyMap(K, d, R, P, size, cv2.CV_32FC1)
        ax, ay = ref_ops.init_undistort_rectify_map(K, d, R, P, size)
        assert np.array_equal(ax, mx) and np.array_equal(ay, my), (size, int((ax != mx).sum()), int((ay != my).sum()))


def test_median_speckles():
    rng = np.random.default_rng(1)
    for t in range(4):
        H, W = (37, 61) if t < 2 else (240, 320)
        d = (rng.integers(-1, 40, (H, W)) * 16 + rng.integers(0, 16, (H, W))).astype(np.int16)
        d[rng.random((H, W)) < 0.3] = -16
        assert np.array_equal(cref.median3_s16(d), cv2.medianBlur(d, 3))
        e = d.copy()
        cv2.filterSpeckles(e, -16, 25, 32)
        assert np.array_equal(cref.filter_speckles(d, -16, 25, 32), e)


def test_simple_masks_and_filters(golden_synth):
    left = golden_synth["left"]
    cfg = dict(hsv_lower=(50, 100, 180), hsv_upper=(70, 255, 255), brightness_threshold=200, min_area=50)
    _, wm1, wm2 = ref_ops.simple_extract(left, want_masks=True, **cfg)
    m1, m2 = cref.simple_masks(left, cfg["hsv_lower"], cfg["hsv_upper"], 200, 50)
    assert np.array_equal(m1, wm1) and np.array_equal(m2, wm2)
    rng = np.random.default_rng(5)
    for t in range(20):  # random blobs: contour semantics (holes, thin bridges, border contact)
        m = (cv2.GaussianBlur(rng.random((60, 80)).astype(np.float32), (0, 0), 1.5 + 0.1 * t) > 0.5).astype(np.uint8) * 255
        img = np.zeros((60, 80, 3), np.uint8)
        img[m > 0] = (140, 255, 140)
        _, wm1, wm2 = ref_ops.simple_extract(img, want_masks=True, **dict(cfg, min_area=8 + t))
        m1, m2 = cref.simple_masks(img, cfg["hsv_lower"], cfg["hsv_upper"], 200, 8 + t)
        assert np.array_equal(m1, wm1) and np.array_equal(m2, wm2), t
    f = cv2.cvtColor(left, cv2.COLOR_BGR2GRAY).astype(np.float32)
    for sigma in (2.0, 3.0):
        # f32 filters: cv2's SIMD summation order is not reproduced -> tolerance 4 ulp of the image range
        assert np.allclose(cref.gaussian_blur_f32(f, sigma), cv2.GaussianBlur(f, (0, 0), sigma), rtol=0, atol=1.3e-4)
    s = cv2.GaussianBlur(f, (0, 0), 3.0)
    for dx, dy in ((1, 0), (0, 1)):
        assert np.allclose(cref.sobel3_f32(s, dx, dy), cv2.Sobel(s, cv2.CV_32F, dx, dy, ksize=3), rtol=0, atol=2e-4)


def test_depth_vs_cv2_real_and_random_Q(golden_real):
    for tag in ("a", "b"):
        assert np.array_equal(cref.disp_to_depth_q(golden_real["disp16_" + tag], golden_real["Q"]), golden_real["depth_" + tag])
    rng = np.random.default_rng(0)
    d16 = rng.integers(-16, 2000, (100, 150)).astype(np.int16)
    Q = np.array([[1, 0, 0, -150.3], [0, 1, 0, -99.7], [0.001, 0.002, 0.0003, 233.123], [0.0001, 0.0002, 16.3, -0.7]])
    assert np.array_equal(cref.disp_to_depth_q(d16, Q), ref_ops.depth_from_disparity(d16, Q))


def test_depth_vs_cv2(golden_synth):
    d16 = golden_synth["disp16_3way"]
    Q = golden_synth["Q"]
    assert np.array_equal(cref.disp_to_depth_q(d16, Q), ref_ops.depth_from_disparity(d16, Q))
    assert np.array_equal(cref.disp_to_depth_q(d16, Q), golden_synth["depth"])
    assert np.array_equal(cref.disp_to_depth_default(d16), ref_ops.depth_from_disparity(d16, None))


def test_wls_restatement_properties():
    """WLS: PARITY UNPINNED (cv2.ximgproc absent).  Check the restatement's invariants only:
    outside-ROI fill, determinism, and that a constant, fully confident field is a fixed point."""
    H, W, D = 40, 120, 32
    guide = np.random.default_rng(0).integers(0, 256, (H, W)).astype(np.uint8)
    dl = np.full((H, W), 10 * 16, np.int16)
    dr = np.full((H, W), -10 * 16, np.int16)
    out, conf = cref.wls_filter(dl, dr, guide, 0, D, 3, want_conf=True)
    assert np.all(out[:, :D] == -16)
    assert np.all(out[:, D + 12:] == 160)
    assert conf.max() <= 255.0 + 1e-3
    assert np.array_equal(out, cref.wls_filter(dl, dr, guide, 0, D, 3))


def wls_case(W, H, D, seed):
    """left/right disparity maps that are mostly LR-consistent (so the confidence is not zero everywhere): a constant
    patch at 587/16 px (in f32 its box variance rounds to -0.03, confidence 1.00003), a smooth ramp with a little noise,
    some invalid pixels, and the invalid borders a real matcher pair leaves outside the two ROIs"""
    rng = np.random.default_rng(seed)
    guide = cv2.GaussianBlur(rng.integers(0, 256, (H, W), dtype=np.uint8), (0, 0), 1.2)
    x = np.arange(W)[None, :].repeat(H, 0)
    d = np.where(x < W // 2, 587, 6 * 16 + (x - W // 2) * 2).astype(np.int32)
    dl = (d + np.where(x < W // 2, 0, rng.integers(-3, 4, (H, W)))).astype(np.int16)
    dl[rng.random((H, W)) < 0.03] = -16
    dl[:, :D] = -16
    dr = (-d + rng.integers(-3, 4, (H, W))).astype(np.int16)
    dr[:, : W // 2] = -587
    dr[:, W - D:] = -16 * D
    return dl, dr, guide


def test_wls_oracle_variants_switch_one_point_each():
    """oracle/csrc/orc_wls.c: the unpinned points of the restatement (SURVEY A7) are switchable; variant 0 is the legacy entry
    point, and every bit changes the result on an input built to exercise it."""
    from oracle import cref
    W, H, D = 150, 33, 48
    dl, dr, guide = wls_case(W, H, D, 3)
    base, bconf = cref.wls_filter(dl, dr, guide, 0, D, 3, 8000.0, 1.5, want_conf=True)
    assert base.shape == (H, W) and (base[:, :D] == -16).all()
    outs = {}
    for bit in (1, 2, 4, 8):
        o, c = cref.wls_filter(dl, dr, guide, 0, D, 3, 8000.0, 1.5, want_conf=True, variant=bit)
        assert not np.array_equal(o, base), "variant bit %d had no effect" % bit
        outs[bit] = o
        if bit == 1:
            assert np.array_equal(c, bconf)  # lambda schedule: the confidence map is untouched
    assert not np.array_equal(outs[2], outs[8])


def test_oracle_on_stored_real_pairs(golden_real, golden_real_more):
    """SURVEY 8c pin (ii): the six of the reference's 28 calibration pairs the goldens store (real_pair_[a-f].npz),
    rectified with the shipped calibration -- the oracle's remap / gray / StereoSGBM restatements against the cv2 binary
    (as constructed: SGBM_3WAY, 64 / 5; and the WLS-mutated left + right matcher pair in MODE_HH), and the goldens the
    REAL camera class produced against what the same cv2 calls produce today."""
    import zlib
    g = golden_real
    size = (320, 240)
    R1, R2, P1, P2, Q, _, _ = cv2.stereoRectify(g["K_left"], g["dist_left"], g["K_right"], g["dist_right"], size,
                                                g["R"], g["T"], flags=cv2.CALIB_ZERO_DISPARITY, alpha=0)
    mlx, mly = cv2.initUndistortRectifyMap(g["K_left"], g["dist_left"], R1, P1, size, cv2.CV_32FC1)
    mrx, mry = cv2.initUndistortRectifyMap(g["K_right"], g["dist_right"], R2, P2, size, cv2.CV_32FC1)
    base, mut, right = ref_ops.sgbm_param_sets(64, 5, 2)
    _, mut_hh, right_hh = ref_ops.sgbm_param_sets(64, 5, 1)
    more = golden_real_more
    for t in ("a", "b", "c", "d", "e", "f"):
        src = g if t in ("a", "b") else more
        frame = src["frame_" + t]
        l, r = np.ascontiguousarray(frame[:, :320]), np.ascontiguousarray(frame[:, 320:])
        lrect, rrect = cv2.remap(l, mlx, mly, cv2.INTER_LINEAR), cv2.remap(r, mrx, mry, cv2.INTER_LINEAR)
        assert np.array_equal(cref.remap_bilinear(l, mlx, mly), lrect), t
        assert np.array_equal(cref.remap_bilinear(r, mrx, mry), rrect), t
        lg, rg = cv2.cvtColor(lrect, cv2.COLOR_BGR2GRAY), cv2.cvtColor(rrect, cv2.COLOR_BGR2GRAY)
        assert np.array_equal(cref.bgr2gray(lrect), lg) and np.array_equal(cref.bgr2gray(rrect), rg), t
        want = cv2.StereoSGBM_create(**base).compute(lg, rg)
        assert np.array_equal(cref.sgbm_compute(lg, rg, **base), want), t
        assert np.array_equal(cref.sgbm_compute(lg, rg, **mut_hh), cv2.StereoSGBM_create(**mut_hh).compute(lg, rg)), t
        assert np.array_equal(cref.sgbm_compute(rg, lg, **right_hh), cv2.StereoSGBM_create(**right_hh).compute(rg, lg)), t
        # the stored golden of this pair is what the calls above produce
        assert np.array_equal(src["disp16_" + t], want), t
        if t in ("a", "b"):
            assert np.array_equal(src["lrect_" + t], lrect) and np.array_equal(src["rrect_" + t], rrect), t
        else:
            assert int(src["lrect_crc_" + t]) == zlib.crc32(lrect.tobytes()), t
            assert int(src["rrect_crc_" + t]) == zlib.crc32(rrect.tobytes()), t


def test_stereo_rectify_vs_cv2(golden_real):
    """SURVEY 8f N3: cv2.stereoRectify restated on the host (camera/rectify.py; reference call
    camera/single_usb_stereo_camera.py:176-187).  On the shipped calibration P1, P2, Q and both ROIs equal cv2 4.x bit for
    bit at every alpha; R1 / R2 differ by at most the last bits (OpenCV re-orthogonalises R with its own Jacobi SVD) and
    the f32 rectification maps built from them are identical.  Synthetic rigs (horizontal / vertical baselines, 5 and 8
    distortion coefficients, with and without CALIB_ZERO_DISPARITY): <= 1e-12 relative, ROIs equal."""
    from laser_3d_reconstruction_b200.camera.rectify import stereo_rectify
    g = golden_real
    K1, d1, K2, d2, R, T = g["K_left"], g["dist_left"], g["K_right"], g["dist_right"], g["R"], g["T"]

    def rel(a, b):
        return float(np.abs(np.asarray(a) - np.asarray(b)).max() / np.abs(np.asarray(b)).max())

    for size in ((320, 240), (640, 480)):
        for alpha in (0, -1, 1, 0.5):
            want = cv2.stereoRectify(K1, d1, K2, d2, size, R, T, flags=cv2.CALIB_ZERO_DISPARITY, alpha=alpha)
            got = stereo_rectify(K1, d1, K2, d2, size, R, T, flags=cv2.CALIB_ZERO_DISPARITY, alpha=alpha)
            assert rel(got[0], want[0]) < 1e-15 and rel(got[1], want[1]) < 1e-15
            assert all(rel(got[i], want[i]) < 1e-14 for i in (2, 3, 4))
            assert got[5] == tuple(want[5]) and got[6] == tuple(want[6])
            if alpha == 0:  # the reference's call
                assert all(np.array_equal(got[i], want[i]) for i in (2, 3, 4)), "P1, P2, Q bit-identical"
                for K, d, Rg, Rw, Pg, Pw in ((K1, d1, got[0], want[0], got[2], want[2]), (K2, d2, got[1], want[1], got[3], want[3])):
                    a = cv2.initUndistortRectifyMap(K, d, Rg, Pg, size, cv2.CV_32FC1)
                    b = cv2.initUndistortRectifyMap(K, d, Rw, Pw, size, cv2.CV_32FC1)
                    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    rng = np.random.default_rng(0)
    for trial in range(8):
        f = 300 + rng.random() * 200
        Ka = np.array([[f, 0, 160 + rng.normal() * 5], [0, f * 1.01, 120 + rng.normal() * 5], [0, 0, 1]])
        Kb = Ka.copy(); Kb[0, 0] *= 1.02; Kb[0, 2] += 3
        da, db = rng.normal(0, 0.02, (1, 5 if trial % 2 else 8)), rng.normal(0, 0.02, (1, 5 if trial % 2 else 8))
        Rm = cv2.Rodrigues(rng.normal(0, 0.02, 3))[0]
        Tm = np.array([[-0.06], [0.002], [0.001]]) if trial < 5 else np.array([[0.001], [-0.05], [0.002]])
        fl = cv2.CALIB_ZERO_DISPARITY if trial % 3 else 0
        want = cv2.stereoRectify(Ka, da, Kb, db, (320, 240), Rm, Tm, flags=fl, alpha=0)
        got = stereo_rectify(Ka, da, Kb, db, (320, 240), Rm, Tm, flags=fl, alpha=0)
        assert all(rel(got[i], want[i]) < 1e-12 for i in range(5)), trial
        assert got[5] == tuple(want[5]) and got[6] == tuple(want[6])


def test_stereo_rectify_random_rigs_vs_cv2():
    """Random rigs (4 .. 14 distortion coefficients incl. the tilted-sensor pair, both baseline directions, every alpha,
    strong distortion that folds inside the image): matrices <= 1e-11 relative, ROIs equal -- except at alpha = 0, where
    an ROI edge sits exactly on the image border and the last bits of R1 / R2 decide between 0 and 1 (camera/rectify.py)."""
    from laser_3d_reconstruction_b200.camera.rectify import stereo_rectify
    rng = np.random.default_rng(11)
    for it in range(60):
        W, H = int(rng.choice([320, 640, 1280])), int(rng.choice([240, 480, 720]))
        f = rng.uniform(0.6, 1.4) * W
        Ks = [np.array([[f * rng.uniform(.97, 1.03), 0, W / 2 + rng.uniform(-20, 20)],
                        [0, f * rng.uniform(.97, 1.03), H / 2 + rng.uniform(-20, 20)], [0, 0, 1]]) for _ in range(2)]
        nd = int(rng.choice([4, 5, 8, 12, 14]))
        ds = []
        for _ in range(2):
            d = np.zeros(nd)
            d[0], d[1] = rng.uniform(-.3, .2), rng.uniform(-.1, .1)
            d[2:4] = rng.uniform(-2e-3, 2e-3, 2)
            if nd > 4:
                d[4] = rng.uniform(-.05, .05)
            if nd >= 8:
                d[5:8] = rng.uniform(-.02, .02, 3)
            if nd >= 12:
                d[8:12] = rng.uniform(-1e-3, 1e-3, 4)
            if nd >= 14:
                d[12:14] = rng.uniform(-1e-2, 1e-2, 2)
            ds.append(d)
        R = cv2.Rodrigues(rng.uniform(-0.05, 0.05, 3))[0]
        T = np.array([-rng.uniform(0.03, 0.2), rng.uniform(-0.005, 0.005), rng.uniform(-0.005, 0.005)])
        if rng.random() < 0.25:
            T = T[[1, 0, 2]]
        flags = int(rng.choice([cv2.CALIB_ZERO_DISPARITY, 0]))
        alpha = float(rng.choice([0, -1, 1, 0.5, 0.25]))
        want = cv2.stereoRectify(Ks[0], ds[0], Ks[1], ds[1], (W, H), R, T, flags=flags, alpha=alpha)
        got = stereo_rectify(Ks[0], ds[0], Ks[1], ds[1], (W, H), R, T, flags=flags, alpha=alpha)
        for i in range(5):
            if np.all(np.isfinite(want[i])):
                assert np.abs(got[i] - want[i]).max() <= 1e-11 * max(np.abs(want[i]).max(), 1.0), (it, i)
            else:
                assert np.array_equal(np.isfinite(got[i]), np.isfinite(want[i])), (it, i)
        for a, b in ((got[5], want[5]), (got[6], want[6])):
            if alpha == 0:
                assert all(abs(int(p) - int(q)) <= 1 for p, q in zip(a, b)), (it, a, tuple(b))
            else:
                assert tuple(a) == tuple(b), (it, a, tuple(b))


def test_sgbm_random_parameter_sets_vs_cv2():
    """A fixed-seed slice of tests/fuzz/fuzz_oracle.py: random StereoSGBM parameter sets (all modes, both disparity signs, odd
    penalties, preFilterCap / uniqueness / disp12MaxDiff / speckle settings) on random small images, oracle == cv2."""
    rng = np.random.default_rng(2024)
    for it in range(24):
        D = int(rng.choice([16, 32, 48, 64, 96, 128]))
        bs = int(rng.choice([1, 3, 5, 7, 9, 11]))
        W, H = int(rng.integers(D + 20, D + 160)), int(rng.integers(8, 60))
        minD = int(rng.choice([0, 0, -(D - 1), 3, -5, 16, -D // 2]))
        P1 = int(rng.choice([24 * bs * bs, 8 * bs * bs, 10, 0, 100]))
        P2 = max(int(rng.choice([96 * bs * bs, 32 * bs * bs, 200, 1000])), P1 + 1)
        kw = dict(minDisparity=minD, numDisparities=D, blockSize=bs, P1=P1, P2=P2, disp12MaxDiff=int(rng.choice([1, 0, -1, 2, 1000000, 5])),
                  preFilterCap=int(rng.choice([63, 63, 31, 15, 1, 40])), uniquenessRatio=int(rng.choice([0, 10, 5, 15, 40])),
                  speckleWindowSize=int(rng.choice([0, 100, 20, 200])), speckleRange=int(rng.choice([32, 1, 2, 16])),
                  mode=int(rng.integers(0, 4)))
        lg, rg = gray_pair(W, H, max(D, 16), int(rng.integers(0, 1000)), quant=int(rng.choice([0, 0, 8, 32])))
        if rng.random() < 0.2:
            lg, rg = rng.integers(0, 256, lg.shape, dtype=np.uint8), rng.integers(0, 256, rg.shape, dtype=np.uint8)
        assert np.array_equal(cref.sgbm_compute(lg, rg, **kw), cv2.StereoSGBM_create(**kw).compute(lg, rg)), (it, W, H, kw)


def test_wls_solver_against_an_independent_f64_solve():
    """The unpinned WLS restatement at least solves the system it claims to: with the oracle's own confidence map as input,
    three iterations of (I + lambda_t L_h) then (I + lambda_t L_v) solved per line in float64 by scipy's banded solver (L =
    weighted graph Laplacian, weights exp(-|dg| / sigma_color), lambda_t = lambda / 4^t) give the oracle's int16 output
    within 1 LSB everywhere and identically on > 99 % of the ROI.  (What stays unpinned is ximgproc's choice of these
    ingredients, not the arithmetic.)"""
    W, H, D = 150, 33, 48
    lam0, sigma = 8000.0, 1.5
    for seed in (3, 8):
        dl, dr, guide = wls_case(W, H, D, seed)
        out, conf = cref.wls_filter(dl, dr, guide, 0, D, 3, lam0, sigma, want_conf=True)
        x0, w, h = D, W - D, H
        g = guide[:, x0:].astype(np.float64)
        wh = np.zeros((h, w)); wv = np.zeros((h, w))
        wh[:, :-1] = np.exp(-np.abs(g[:, :-1] - g[:, 1:]) / sigma)
        wv[:-1, :] = np.exp(-np.abs(g[:-1, :] - g[1:, :]) / sigma)
        c = conf[:, x0:].astype(np.float64)
        num, den = ref_ops.fgs_f64(c * dl[:, x0:].astype(np.float64), c, -wh, -wv, lam0, 3)
        want = np.clip(np.rint(num / (den + 1e-43)), -32768, 32767)
        got = out[:, x0:].astype(np.float64)
        diff = np.abs(got - want)
        assert diff.max() <= 1, diff.max()
        assert (diff == 0).mean() > 0.99, (diff == 0).mean()


@pytest.mark.parametrize("variant", [0, 1, 15])
def test_fgs_f32_restatement_reproduces_the_oracle(variant):
    """ref_ops.fgs_f32_serial (numpy float32, vectorised over lines) repeats orc_wls.c's fgs_solve operation for operation:
    fed the oracle's own confidence map and guide weights, it gives the oracle's int16 output bit for bit, under either
    lambda schedule.  The GPU solver tests measure the serial f32 error with it, so it must not be an unchecked helper."""
    lam0, sigma = 8000.0, 1.5
    for (W, H, D), seed in (((150, 33, 48), 3), ((97, 40, 16), 8)):
        dl, dr, guide = wls_case(W, H, D, seed)
        out, conf = cref.wls_filter(dl, dr, guide, 0, D, 3, lam0, sigma, want_conf=True, variant=variant)
        x0 = D
        c = conf[:, x0:]
        ch, cv = ref_ops.wls_weights(guide[:, x0:], sigma)
        num, den = ref_ops.fgs_f32_serial(c * dl[:, x0:].astype(np.float32), c, ch, cv, lam0, 3, variant)
        with np.errstate(over="ignore", invalid="ignore"):
            v = num * (np.float32(1) / (den + np.float32(1e-43)))
        q = np.where(np.abs(v) < np.float32(2 ** 31), np.rint(np.nan_to_num(v)), -32768)
        got = np.clip(q, -32768, 32767).astype(np.int16)
        assert np.array_equal(got, out[:, x0:]), "%d of %d pixels differ" % ((got != out[:, x0:]).sum(), got.size)
        assert (out[:, :x0] == -16).all()
