"""The kernels that run on every frame around the matcher, at the shapes and values the benchmark never feeds them:
remap + gray, the Simple and Steger extractors, median / speckles, disparity -> depth, the reconstruction kinds, the
laser depth map, the point-cloud sink past its first scan level and the device packing of the frame pipeline.

Integer stages and stages that claim bit-exactness are compared bit for bit with cv2 or the oracle.  The Steger
variants keep their 0.01 px contract, checked by `steger_mismatch_ok`: each candidate is evaluated in float64 from
cv2's f32 derivative images and from the same images in the GPU's f32 operation order, and a point that only one side
reports is accepted only where those two disagree or a decision lies within a few f32 ulps of its boundary."""
import ctypes as C

import cv2
import numpy as np
import pytest

from laser_3d_reconstruction_b200 import _native as N
from laser_3d_reconstruction_b200 import pipeline, synth
from oracle import ref_ops

pytestmark = pytest.mark.gpu

GREEN = (140, 255, 140)  # inside the Simple extractor's HSV range below, gray 207 > 200
SIMPLE_LO, SIMPLE_HI = (50, 100, 180), (70, 255, 255)


def eq(a, b, what=""):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, "%s: shape %s vs %s" % (what, a.shape, b.shape)
    bad = np.argwhere(~((a == b) | ((a != a) & (b != b))))  # NaN == NaN here: both sides must give NaN
    assert len(bad) == 0, "%s: %d/%d differ, first %s got %s want %s" % (
        what, len(bad), a.size, tuple(bad[0]), a[tuple(bad[0])], b[tuple(bad[0])])


# ---- remap + gray --------------------------------------------------------------------------------------------------
def _special_map(rng, W, H, sw, sh):
    """a random map over [-4, size + 4) with exact fixed-point ties and the taps at the source's edges mixed in"""
    mx = (rng.random((H, W)) * (sw + 8) - 4).astype(np.float32)
    my = (rng.random((H, W)) * (sh + 8) - 4).astype(np.float32)
    specx = np.array([-1 / 64, -1 / 32, -0.5, -1, sw - 1, sw - 1 + 1 / 32, sw - 1 + 1 / 64, 0, 0.5 / 32], np.float32)
    specy = np.array([-1 / 64, -1 / 32, -0.5, -1, sh - 1, sh - 1 + 1 / 32, sh - 1 + 1 / 64, 0, 0.5 / 32], np.float32)
    ties = rng.random((H, W)) < 0.3  # k/64: v * 32 lands on .5, rounded half to even
    mx[ties] = np.round(mx[ties] * 64) / 64
    my[ties] = np.round(my[ties] * 64) / 64
    sel = rng.random((H, W)) < 0.3
    mx[sel] = rng.choice(specx, int(sel.sum()))
    sel = rng.random((H, W)) < 0.3
    my[sel] = rng.choice(specy, int(sel.sum()))
    return mx, my


def _remap_check(ctx, src, mx, my, what):
    H, W = mx.shape
    ctx.set_rectify_maps(0, mx, my)
    rect, gray = ctx.remap_gray(0, src, (H, W))
    want = cv2.remap(np.ascontiguousarray(src), mx, my, cv2.INTER_LINEAR)
    eq(rect, want, what + " rect")
    eq(gray, cv2.cvtColor(want, cv2.COLOR_BGR2GRAY), what + " gray")


@pytest.mark.parametrize("H", [1, 2, 1027])
@pytest.mark.parametrize("W", [1, 2, 3, 5, 127, 129, 1283])
def test_remap_shapes_and_edge_taps(ctx, W, H):
    """Widths that are not a multiple of 4, so every row ends in the byte-store tail (1-5: only the tail); the vector
    store path is covered by test_remap_vector_store_widths.  1027 rows exercise the grid's y extent.  Sources
    smaller, equal and larger than the map, and a side-by-side view with a row stride of twice its width."""
    rng = np.random.default_rng(W * 7919 + H)
    for sw, sh in ((max(W // 2, 1), max(H // 2, 1)), (W, H), (2 * W + 3, H + 5)):
        src = rng.integers(0, 256, (sh, sw, 3), dtype=np.uint8)
        mx, my = _special_map(rng, W, H, sw, sh)
        _remap_check(ctx, src, mx, my, "%dx%d from %dx%d" % (W, H, sw, sh))
    frame = rng.integers(0, 256, (H, 2 * W, 3), dtype=np.uint8)
    mx, my = _special_map(rng, W, H, W, H)
    _remap_check(ctx, frame[:, W:], mx, my, "side-by-side view")


def test_remap_vector_store_widths(ctx):
    """W % 4 == 0: the 12 + 4 byte vector stores, next to W % 4 != 0 of the same height"""
    rng = np.random.default_rng(4)
    for W in (4, 128, 1280, 1284):
        src = rng.integers(0, 256, (37, W, 3), dtype=np.uint8)
        mx, my = _special_map(rng, W, 37, W, 37)
        _remap_check(ctx, src, mx, my, "W=%d" % W)


def _nonfinite_maps(rng, W, H, vals, where):
    mx, my = _special_map(rng, W, H, W, H)
    for v in vals:
        sel = rng.random((H, W)) < 0.03
        if where in ("x", "both"):
            mx[sel] = v
        if where in ("y", "both"):
            my[sel] = v
    return mx, my


@pytest.mark.parametrize("where", ["x", "y", "both"])
def test_remap_nan_map_entries_sample_the_border(ctx, where):
    """cv2 rounds a NaN map entry to INT_MIN (cvRound) and samples the constant border 0; the library must too --
    cvt.rni alone turns NaN into 0 and samples source pixel 0 of that axis"""
    rng = np.random.default_rng({"x": 1, "y": 2, "both": 3}[where])
    for W, H in ((97, 53), (320, 240)):
        src = rng.integers(1, 256, (H, W, 3), dtype=np.uint8)  # no zero pixel: a wrong tap cannot hide
        mx, my = _nonfinite_maps(rng, W, H, [np.nan], where)
        _remap_check(ctx, src, mx, my, "NaN in %s" % where)


@pytest.mark.parametrize("where", ["x", "y", "both"])
def test_remap_infinite_and_huge_map_entries(ctx, where):
    rng = np.random.default_rng({"x": 4, "y": 5, "both": 6}[where])
    W, H = 129, 61
    src = rng.integers(1, 256, (H, W, 3), dtype=np.uint8)
    mx, my = _nonfinite_maps(rng, W, H, [np.inf, -np.inf, 3e9, -3e9, 1e6, -1e6, 3.4e38, -3.4e38], where)
    _remap_check(ctx, src, mx, my, "non-finite / huge in %s" % where)


def _nan_rig(W, H, D):
    K, Q = synth.camera_model(W, H)
    maps = list(synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1))
    rng = np.random.default_rng(11)
    mx, my = maps[0].copy(), maps[1].copy()
    mx[:, :17] = np.nan  # a band the left matcher sees as border, plus scattered holes in both maps
    mx[rng.random((H, W)) < 0.01] = np.nan
    my[rng.random((H, W)) < 0.01] = np.nan
    maps[0], maps[1] = mx, my
    return K, Q, maps


def test_compute_depth_and_pipeline_with_partly_nan_left_map(ctx):
    """A degenerate rig (stereo_rectify returns NaN matrices) or a user's own maps give NaN entries: the rectified
    view and everything after it must still follow the reference computed with the same maps"""
    W, H, D, bs, mode = 320, 360, 64, 5, 2
    K, Q, maps = _nan_rig(W, H, D)
    left, right = synth.stereo_pair(W, H, D, 4)
    wrect, wdepth, aux = ref_ops.depth_path(left, right, maps, D, bs, mode, Q, want_all=True)
    ctx.set_rectify_maps(0, maps[0], maps[1])
    ctx.set_rectify_maps(1, maps[2], maps[3])
    rect, depth, disp = ctx.compute_depth(pipeline.depth_config(D, bs, mode, Q), left, right, want_disp=True)
    eq(rect, wrect, "compute_depth rect")
    diff = np.abs(disp.astype(np.int32) - aux["df"].astype(np.int32))
    assert (diff <= 1).mean() >= 0.999, "compute_depth disparity: %.5f within 1 LSB" % (diff <= 1).mean()
    cfg = pipeline.make_pipeline_config(W, H, D, bs, mode, Q, K, lanes=1, max_points=8000)
    fp = pipeline.FramePipeline(cfg, maps=maps, ctx=ctx)
    try:
        fp.run_host(left[None].copy(), right[None].copy())
        got = fp.fetch(0)
    finally:
        fp.close()
    eq(got["left_rect"], wrect, "pipeline rect")
    diff = np.abs(got["disp16"].astype(np.int32) - aux["df"].astype(np.int32))
    assert (diff <= 1).mean() >= 0.999, "pipeline disparity: %.5f within 1 LSB" % (diff <= 1).mean()


# ---- Simple extractor ------------------------------------------------------------------------------------------------
def _simple_check(ctx, img, min_area, what):
    wpts, wm1, wm2 = ref_ops.simple_extract(img, SIMPLE_LO, SIMPLE_HI, 200, min_area, want_masks=True)
    pts, m1, m2 = ctx.simple_extract(img, SIMPLE_LO, SIMPLE_HI, 200, min_area, want_masks=True)
    eq(m1, wm1, what + " morph mask")
    eq(m2, wm2, what + " final mask")
    eq(pts, np.array(wpts, np.float64).reshape(-1, 2), what + " points")
    return pts


@pytest.mark.parametrize("H", [1, 2, 1500])
@pytest.mark.parametrize("W", [1, 2, 129, 1283])
def test_simple_extractor_shapes_and_border_stripes(ctx, W, H):
    """stripes on every border, a diagonal band and blobs; 1500 rows make row_scan_kernel carry across its 1024-row
    blocks"""
    rng = np.random.default_rng(W + 31 * H)
    img = rng.integers(0, 120, (H, W, 3), dtype=np.uint8)
    img[:, :min(4, W)] = GREEN
    img[:, max(W - 5, 0):] = GREEN
    img[:min(3, H)] = GREEN
    img[max(H - 4, 0):] = GREEN
    yy, xx = np.mgrid[0:H, 0:W]
    img[np.abs(xx - 0.7 * yy - W / 3) < 4] = GREEN
    for _ in range(H * W // 20000):
        y, x = rng.integers(0, H), rng.integers(0, W)
        img[y:y + rng.integers(3, 12), x:x + rng.integers(3, 12)] = GREEN
    # varying brightness inside the mask, so every row's centroid is a real weighted mean
    g = img.astype(np.int32)
    m = (img == GREEN).all(-1)
    g[m, 1] = 255 - rng.integers(0, 10, int(m.sum()))  # stays inside the HSV range
    pts = _simple_check(ctx, g.astype(np.uint8), 50 if W * H > 200 else 0, "%dx%d" % (W, H))
    if H == 1500 and W >= 129:
        assert len(pts) == H


def test_simple_extractor_diagonal_hole_and_area_threshold(ctx):
    """a hole that reaches the outside only through diagonal steps is filled (the background is 4-connected); blobs
    whose contour area equals min_area are dropped, and kept at min_area - 0.5"""
    img = np.zeros((60, 90, 3), np.uint8)
    img[5:25, 5:10] = GREEN; img[5:10, 5:25] = GREEN  # two thick Ls touching at two corners only
    img[10:30, 25:30] = GREEN; img[25:30, 10:30] = GREEN
    img[40:47, 40:52] = GREEN  # 7 x 12: contour area 6 * 11 = 66
    for i in range(10):  # a staircase triangle: contour area 36.5
        img[40 + i, 60:70 - i] = GREEN
    _, m1, m2 = ref_ops.simple_extract(img, SIMPLE_LO, SIMPLE_HI, 200, 0, want_masks=True)
    assert (m2 > 0).sum() == (m1 > 0).sum() + 15 * 15, "the diagonal-only hole must be filled in the reference"
    contours, _ = cv2.findContours(m1, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
    areas = sorted({cv2.contourArea(c) for c in contours})
    assert any(a != int(a) for a in areas)
    for a in areas:
        for min_area in (a, a - 0.5):
            _simple_check(ctx, img, min_area, "min_area %.1f" % min_area)


# ---- Steger ----------------------------------------------------------------------------------------------------------
def steger_params(variant, sigma, roi=(0, 0, 0, 0), bright=200, resp=0.5):
    return N.StegerParams(variant, sigma, bright, resp, (C.c_int * 4)(*roi), (C.c_int * 3)(*SIMPLE_LO),
                          (C.c_int * 3)(*SIMPLE_HI))


def ridge_gray(W, H, period, angle, seed, width=1.3, gain=200):
    """straight bright ridges (Gaussian profile of height `gain`, clipped at 255) over a dim background, at a random
    phase"""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float64)
    d = xx * np.cos(angle) + yy * np.sin(angle) + rng.random() * period
    d = (d % period) - period / 2
    return np.clip(np.rint(50 + gain * np.exp(-d * d / (2 * width * width))), 0, 255).astype(np.uint8)


def ridge_bgr(gray):
    """green ridges for the Hybrid extractor's HSV range: B = R = 0.6 G"""
    g = gray.astype(np.float64)
    return np.stack([0.6 * g, g, 0.6 * g], -1).round().astype(np.uint8)


def _derivs(variant, img, sigma, roi=None):
    """the oracle's f32 derivative images (dx, dy, dxx, dxy, dyy), its selection image, the ROI offset and the gray
    image the derivatives come from"""
    gray = cv2.cvtColor(img, cv2.COLOR_BGR2GRAY) if img.ndim == 3 else img
    if variant == N.STEGER_FAST:
        ox = oy = 0
        if roi is not None:
            ox, oy, rw, rh = roi
            gray = gray[oy:oy + rh, ox:ox + rw]
        f = cv2.GaussianBlur(gray.astype(np.float32), (0, 0), sigma, sigma)
        k = lambda a: np.array(a, np.float32)
        d = [cv2.filter2D(f, cv2.CV_32F, k(a)) for a in ([[1, -1]], [[1], [-1]], [[1, -2, 1]], [[1, -1], [-1, 1]],
                                                         [[1], [-2], [1]])]
        return d, gray > 200, (ox, oy), gray
    if variant == N.STEGER_HYBRID:
        hsv = cv2.cvtColor(img, cv2.COLOR_BGR2HSV)
        mask = cv2.bitwise_and(cv2.inRange(hsv, np.asarray(SIMPLE_LO), np.asarray(SIMPLE_HI)),
                               (gray > 200).astype(np.uint8) * 255)
        mask = cv2.morphologyEx(cv2.morphologyEx(mask, cv2.MORPH_CLOSE, np.ones((3, 3), np.uint8)), cv2.MORPH_OPEN,
                                np.ones((3, 3), np.uint8))
        roi = img.copy()
        roi[mask == 0] = 0
        gray, sel = cv2.cvtColor(roi, cv2.COLOR_BGR2GRAY), mask > 0
    else:
        sel = gray > 200
    dx, dy, dxx, dyy, dxy = ref_ops._sobel_chain(gray.astype(np.float32), sigma)
    sel = sel.copy()
    sel[[0, -1], :] = False
    sel[:, [0, -1]] = False
    return [dx, dy, dxx, dxy, dyy], sel, (0, 0), gray


def _decide64(variant, d, resp_thr, w, h, xx, yy):
    """the candidate decisions in float64 from derivatives d = (dx, dy, dxx, dxy, dyy), each (..., n) -> (ok, cx, cy,
    response)"""
    dx, dy, a, b, c = d
    hm, hd = 0.5 * (a + c), 0.5 * (a - c)
    rad = np.sqrt(hd * hd + b * b)
    l1, l2 = hm + rad, hm - rad
    lam = np.where(np.abs(l1) >= np.abs(l2), l1, l2)
    v1x, v1y, v2x, v2y = b, lam - a, lam - c, b
    n1, n2 = v1x * v1x + v1y * v1y, v2x * v2x + v2y * v2y
    vx, vy, nn = np.where(n1 >= n2, v1x, v2x), np.where(n1 >= n2, v1y, v2y), np.maximum(n1, n2)
    with np.errstate(all="ignore"):
        nx = np.where(nn > 0, vx / np.sqrt(nn), np.where(np.abs(a) >= np.abs(c), 1.0, 0.0))
        ny = np.where(nn > 0, vy / np.sqrt(nn), np.where(np.abs(a) >= np.abs(c), 0.0, 1.0))
        den = nx * nx * a + 2 * nx * ny * b + ny * ny * c
        t = -(nx * dx + ny * dy) / den
    ox, oy = t * nx, t * ny
    if variant == N.STEGER_FAST:
        ok = (np.abs(den) > 1e-10) & (np.abs(ox) <= 0.5) & (np.abs(oy) <= 0.5)
    else:
        ok = (lam < 0) & (np.abs(den) >= 1e-6)
        ok &= (np.abs(ox) <= 0.5) if variant == N.STEGER_HYBRID else ((np.abs(ox) <= resp_thr) & (np.abs(oy) <= resp_thr))
    cx, cy = xx + ox, yy + oy
    if variant == N.STEGER_IMPROVED:
        ok &= (cx >= 0) & (cx < w) & (cy >= 0) & (cy < h)
    return ok, cx, cy, np.abs(lam)


def _refl(i, n):
    """BORDER_REFLECT_101 indices, reflected as often as needed (images smaller than the Gaussian radius)"""
    i = np.array(i)
    if n == 1:
        return np.zeros_like(i)
    while ((i < 0) | (i >= n)).any():
        i = np.where(i < 0, -i, np.where(i >= n, 2 * n - 2 - i, i))
    return i


def _at(img, dy, dx):
    h, w = img.shape
    return img[_refl(np.arange(h) + dy, h)[:, None], _refl(np.arange(w) + dx, w)[None, :]]


def _gpu_order_derivs(variant, gray, sigma):
    """The derivative images in the GPU kernels' own f32 operation order (csrc/laser.cu: gauss_row_kernel /
    gauss_col_kernel, then hess_diff or hess_sobel; every step there is an __f*_rn intrinsic, so numpy float32
    reproduces it).  They differ from cv2's by its SIMD summation order only, and that difference is the error
    allowance of the mismatch check."""
    f32 = np.float32
    ks = int(np.rint(sigma * 8 + 1)) | 1
    r = ks // 2
    s2 = -0.5 / (sigma * sigma)
    kd = [np.exp(s2 * (i - r) * (i - r)) for i in range(ks)]
    tot = 0.0
    for v in kd:
        tot += v
    k = np.array([v / tot for v in kd], f32)
    img = gray.astype(f32)
    for axis in (1, 0):  # row pass, then column pass
        sh = (lambda j: _at(img, 0, j)) if axis == 1 else (lambda j: _at(img, j, 0))
        s = k[r] * img
        for j in range(1, r + 1):
            s = s + k[r + j] * (sh(-j) + sh(j))
        img = s
    I = img
    if variant == N.STEGER_FAST:
        c, l, rr, u, d = I, _at(I, 0, -1), _at(I, 0, 1), _at(I, -1, 0), _at(I, 1, 0)
        m2c = f32(-2) * c
        return [l - c, u - c, (l + m2c) + rr, ((_at(I, -1, -1) - u) - l) + c, (u + m2c) + d]
    sm = lambda a, b, c: (a + c) + f32(2) * b
    sdx = lambda J: sm(_at(J, -1, 1) - _at(J, -1, -1), _at(J, 0, 1) - _at(J, 0, -1), _at(J, 1, 1) - _at(J, 1, -1))
    sdy = lambda J: (sm(_at(J, 1, -1), _at(J, 1, 0), _at(J, 1, 1)) - sm(_at(J, -1, -1), _at(J, -1, 0), _at(J, -1, 1)))
    DX, DY = sdx(I), sdy(I)
    return [DX, DY, sdx(DX), sdy(DX), sdy(DY)]


ULPS = 8  # "a few f32 ulps": the f32 eigen-decomposition and the last roundings of the decision quantities


def _near(q, thr):
    """q within ULPS f32 ulps of the threshold thr"""
    return np.abs(q - thr) <= ULPS * 2.0 ** -23 * np.maximum(np.abs(q), np.abs(thr))


def _flip_margins(variant, d, resp_thr, w, h, xx, yy):
    """(near, possible): near where a decision of the candidate lies within ULPS f32 ulps of its boundary, possible
    where every decision passes or is near (float64 from derivatives d).  An eigenvalue order within ULPS ulps counts
    as both: the other eigenvector decides then."""
    dx, dy, a, b, c = d
    hm, hd = 0.5 * (a + c), 0.5 * (a - c)
    rad = np.sqrt(hd * hd + b * b)
    l1, l2 = hm + rad, hm - rad
    lam = np.where(np.abs(l1) >= np.abs(l2), l1, l2)
    _, cx, cy, _ = _decide64(variant, d, resp_thr, w, h, xx, yy)
    ox, oy = cx - xx, cy - yy
    with np.errstate(all="ignore"):
        nx, ny = np.where(np.abs(ox) + np.abs(oy) > 0, ox, 1.0), oy  # direction of the offset = +-n
        nn = np.sqrt(nx * nx + ny * ny)
        nx, ny = nx / nn, ny / nn
        den = nx * nx * a + 2 * nx * ny * b + ny * ny * c
    tests = []  # (passes, near) per decision
    thr = 0.5 if variant in (N.STEGER_FAST, N.STEGER_HYBRID) else resp_thr
    tests.append((np.abs(ox) <= thr, _near(np.abs(ox), thr)))
    if variant != N.STEGER_HYBRID:
        tests.append((np.abs(oy) <= thr, _near(np.abs(oy), thr)))
    if variant == N.STEGER_FAST:
        tests.append((np.abs(den) > 1e-10, _near(np.abs(den), 1e-10)))
    else:
        tests.append((lam < 0, np.abs(lam) <= ULPS * 2.0 ** -23 * (np.abs(a) + np.abs(b) + np.abs(c))))
        tests.append((np.abs(den) >= 1e-6, _near(np.abs(den), 1e-6)))
    if variant == N.STEGER_IMPROVED:
        tests += [(cx >= 0, _near(cx, 0)), (cx < w, _near(cx, w)), (cy >= 0, _near(cy, 0)), (cy < h, _near(cy, h))]
    eig = _near(np.abs(l1), np.abs(l2))
    near = eig | np.any([m for _, m in tests], 0)
    possible = eig | np.all([p | m for p, m in tests], 0)
    return near, possible


def steger_mismatch_ok(variant, img, sigma, got, want, resp_thr=0.5, roi=None, tol=0.01, what=""):
    """The Steger contract: the two point sets pair up within tol = 0.01 px.  Each candidate pixel is evaluated in
    float64 twice, from cv2's f32 derivative images and from the same images in the GPU's f32 operation order.
      * A point pairs within tol plus the distance between the candidate's two float64 points (the part of the
        position that the f32 summation order alone decides).
      * A point that one side has and the other lacks is accepted only if its candidate's decision differs between
        the two derivative sets, or one of its decisions (eigenvalue order, lambda sign, |den|, |t n| and the image
        bounds) lies within ULPS f32 ulps of its boundary under either set.  For the per-row-best variants, the row's
        winner must be contested: two candidates whose responses are within ULPS ulps, or different winners under the
        two sets.
    Any other mismatch fails.  Returns the number of accepted mismatches."""
    got, want = np.asarray(got, np.float64).reshape(-1, 2), np.asarray(want, np.float64).reshape(-1, 2)
    d_cv, sel, (ox, oy), gray = _derivs(variant, img, sigma, roi)
    d_gpu = _gpu_order_derivs(variant, gray, sigma)
    h, w = sel.shape
    yy, xx = np.nonzero(sel)
    fx, fy = xx.astype(np.float64), yy.astype(np.float64)
    per_row = variant in (N.STEGER_OPTIMIZED, N.STEGER_HYBRID)
    ev = []
    for d in (d_cv, d_gpu):
        dv = [di[yy, xx].astype(np.float64) for di in d]
        ok, cx, cy, resp = _decide64(variant, dv, resp_thr, w, h, fx, fy)
        if per_row:  # their points sit on the row itself
            cy = fy.copy()
        ev.append((ok, cx + ox, cy + oy, resp) + _flip_margins(variant, dv, resp_thr, w, h, fx, fy))
    (ok0, cx0, cy0, r0, m0, p0), (ok1, cx1, cy1, r1, m1, p1) = ev
    spread = np.maximum(np.abs(cx0 - cx1), np.abs(cy0 - cy1))
    ambiguous = (ok0 != ok1) | (m0 & p0) | (m1 & p1)
    if per_row:
        contested = np.zeros(h, bool)
        for ok, resp in ((ok0, r0), (ok1, r1)):
            top = np.full(h, -np.inf)
            np.maximum.at(top, yy[ok], resp[ok])
            close = ok & (resp >= top[yy] * (1 - ULPS * 2.0 ** -23))
            contested |= np.bincount(yy[close], minlength=h) > 1
        wins = []
        for ok, resp in ((ok0, r0), (ok1, r1)):  # each set's winner per row: highest response, then lowest x
            win = np.full(h, -1)
            for i in np.argsort(-np.where(ok, resp, -np.inf), kind="stable")[::-1]:
                if ok[i]:
                    win[yy[i]] = i
            wins.append(win)
        contested |= wins[0] != wins[1]
        ambiguous |= (ok0 | ok1) & contested[yy]
    # candidate of a point: a pixel within one of it whose float64 point (either set) lies on it, within its spread
    pts = np.concatenate([got, want])
    side = np.r_[np.zeros(len(got), bool), np.ones(len(want), bool)]
    bad, accepted = [], 0
    for p, is_want in zip(pts, side):
        other = got if is_want else want
        near = np.flatnonzero((np.abs(fx + ox - p[0]) <= 1) & (np.abs(fy + oy - p[1]) <= 1) &
                              (np.minimum(np.hypot(cx0 - p[0], cy0 - p[1]), np.hypot(cx1 - p[0], cy1 - p[1])) <=
                               tol + spread + 1e-5))
        lim = tol + (spread[near].max() if len(near) else 0.0)
        if len(other) and np.hypot(other[:, 0] - p[0], other[:, 1] - p[1]).min() <= lim:
            continue
        if len(near) and ambiguous[near].any():
            accepted += 1
        else:
            bad.append(tuple(p))
            if len(bad) >= 20:
                break
    assert not bad, "%s variant %d: %d lone points with a clear margin, first %s (got %d, want %d points)" % (
        what, variant, len(bad), bad[0], len(got), len(want))
    return accepted


REFS = {N.STEGER_FAST: lambda img, s, roi=None: ref_ops.fast_steger_extract(img, s, 200, roi),
        N.STEGER_IMPROVED: lambda img, s, roi=None: ref_ops.improved_steger_extract(img, s, 200, 0.5),
        N.STEGER_OPTIMIZED: lambda img, s, roi=None: ref_ops.improved_steger_extract_optimized(img, s, 200, 0.5),
        N.STEGER_HYBRID: lambda img, s, roi=None: ref_ops.hybrid_extract(img, SIMPLE_LO, SIMPLE_HI, 200, s)}


def _steger_check(ctx, variant, img, sigma, roi=(0, 0, 0, 0), what=""):
    r = tuple(roi) if roi[2] > 0 and roi[3] > 0 else None
    got = ctx.steger_extract(steger_params(variant, sigma, roi), img)
    want = np.array(REFS[variant](img, sigma, r), np.float64).reshape(-1, 2)
    assert len(want) > 0, "%s variant %d: the reference finds no points" % (what, variant)
    steger_mismatch_ok(variant, img, sigma, got, want, roi=r, what=what)
    return got, want


STEGER_SHAPES = [(5, 300, 16.0), (300, 5, 16.0), (255, 64, 3.0), (256, 64, 8.0), (257, 64, 0.5), (300, 31, 3.0),
                 (300, 32, 8.0), (300, 33, 0.5), (160, 1025, 3.0), (1283, 40, 16.0)]


@pytest.mark.parametrize("W,H,sigma", STEGER_SHAPES)
def test_steger_shapes_and_sigmas(ctx, W, H, sigma):
    """images narrower / shorter than the Gaussian radius (several reflections), widths around the 256-column row
    segments, heights around the 32-row column tiles and past the scan's 1024-row block; sigma 0.5 to 16 (129 taps).
    The grating's period grows with sigma so that its contrast survives the blur.  The Hybrid image's ridges are
    flat-topped and wide, so its colour mask keeps several pixels per row through the 3x3 opening, and the reference
    finds a point in nearly every row the mask reaches."""
    seed = W * 131 + H
    period, angle = max(9.0, 6 * sigma), 0.35 + 0.01 * (seed % 50)
    gray = ridge_gray(W, H, period, angle, seed, width=max(1.3, 0.4 * sigma))
    what = "%dx%d sigma %.1f" % (W, H, sigma)
    for variant in (N.STEGER_FAST, N.STEGER_IMPROVED, N.STEGER_OPTIMIZED):
        _steger_check(ctx, variant, gray, sigma, what=what + " gray")
    _steger_check(ctx, N.STEGER_FAST, ridge_bgr(gray), sigma, what=what + " bgr")
    bgr = ridge_bgr(ridge_gray(W, H, period, angle, seed, width=max(3.0, 0.4 * sigma), gain=300))
    _, want = _steger_check(ctx, N.STEGER_HYBRID, bgr, sigma, what=what + " hybrid")
    rows = np.unique(np.nonzero(_derivs(N.STEGER_HYBRID, bgr, sigma)[1])[0])
    assert len(rows) >= 3 and len(want) >= 0.9 * len(rows), "%s: hybrid %d points, mask in %d rows" % (
        what, len(want), len(rows))


def test_steger_sigma_limit(ctx):
    gray = ridge_gray(64, 48, 9.0, 0.4, 1)
    ctx.steger_extract(steger_params(N.STEGER_FAST, 16.0), gray)  # ks 129: accepted
    with pytest.raises(N.L3DError, match=r"\(-1\).*sigma too large"):  # ks 131
        ctx.steger_extract(steger_params(N.STEGER_FAST, 16.2), gray)


def test_fast_steger_roi_edges(ctx):
    """ROI flush with each edge, past the right / bottom edge (numpy's slice clips it) and wholly outside.  There the
    reference slices an empty image and cv2.GaussianBlur raises; the library documents an empty ROI as no points."""
    W, H = 200, 150
    gray = ridge_gray(W, H, 11.0, 0.5, 3)
    for roi in ((0, 0, 60, 150), (140, 0, 60, 150), (0, 0, 200, 40), (0, 110, 200, 40), (150, 100, 80, 90),
                (170, 20, 500, 30), (10, 140, 40, 500)):
        got, want = _steger_check(ctx, N.STEGER_FAST, gray, 3.0, roi, "roi %s" % (roi,))
        assert len(want) > 0
    for roi in ((200, 0, 10, 10), (0, 150, 10, 10), (500, 400, 30, 30)):
        with pytest.raises(cv2.error):
            ref_ops.fast_steger_extract(gray, 3.0, 200, roi)
        assert len(ctx.steger_extract(steger_params(N.STEGER_FAST, 3.0, roi), gray)) == 0


@pytest.mark.parametrize("dx", [40, 200])
def test_per_row_best_ties_keep_the_lower_x(ctx, dx):
    """two identical vertical ridges in every row: away from the borders their responses are bit-identical, and the
    reference's np.argmax and the GPU's key both keep the lower x.  dx 40: both in one 128-column chunk; 200: in
    different chunks.  The GPU's row winner must be, bit for bit, its point on an image with the left ridge alone."""
    W, H, x0 = 400, 48, 60.0  # three pixels above the Hybrid mask's thresholds survive its 3x3 opening
    xx = np.arange(W, dtype=np.float64)
    prof = lambda c: np.exp(-(xx - c) ** 2 / (2 * 3.0 ** 2))
    one = np.rint(50 + 205 * prof(x0)).astype(np.uint8)
    two = np.rint(50 + 205 * np.maximum(prof(x0), prof(x0 + dx))).astype(np.uint8)
    assert np.array_equal(two[int(x0) - 8:int(x0) + 9], two[int(x0) + dx - 8:int(x0) + dx + 9])
    for variant in (N.STEGER_OPTIMIZED, N.STEGER_HYBRID):
        imgs = [np.repeat(r[None], H, 0) for r in (one, two)]
        if variant == N.STEGER_HYBRID:
            imgs = [ridge_bgr(i) for i in imgs]
        d, sel, _, _ = _derivs(variant, imgs[1], 2.0)
        lam = _decide64(variant, [di[H // 2].astype(np.float64) for di in d], 0.5, W, H, xx, float(H // 2))[3]
        pk = [int(np.argmax(np.where(sel[H // 2] & (np.abs(xx - c) < 3), lam, -1))) for c in (x0, x0 + dx)]
        assert lam[pk[0]] == lam[pk[1]], "the oracle's two ridge responses must tie exactly"
        want = np.array(REFS[variant](imgs[1], 2.0), np.float64).reshape(-1, 2)
        assert len(want) == H - 2 and (want[:, 0] < x0 + 1).all(), "reference keeps the first maximum"
        alone = ctx.steger_extract(steger_params(variant, 2.0), imgs[0])
        got = ctx.steger_extract(steger_params(variant, 2.0), imgs[1])
        assert got.shape == (H - 2, 2) and np.array_equal(got, alone), "variant %d: the lower-x ridge must win" % variant
        assert np.abs(got - want).max() <= 0.01


def test_fast_steger_capacity_rerun(ctx):
    """a fine grating gives more points than the first capacity guess 4 max(W, H) + 4096: the wrapper reruns with the
    reported count, and the result equals one run with room to spare"""
    W, H = 400, 400
    gray = ridge_gray(W, H, 4.0, 0.05, 9, width=0.9)
    got = ctx.steger_extract(steger_params(N.STEGER_FAST, 0.5), gray)
    assert len(got) > 4 * max(W, H) + 4096
    cap = len(got) + 100
    xy = np.empty((cap, 2), np.float32)
    n = C.c_int(0)
    ctx.check(ctx.lib.l3d_steger_extract(ctx.h, C.byref(steger_params(N.STEGER_FAST, 0.5)), gray.ctypes.data_as(C.c_void_p),
                                         1, W, H, xy.ctypes.data_as(C.c_void_p), cap, C.byref(n)), "l3d_steger_extract")
    assert n.value == len(got) and np.array_equal(xy[:n.value], got)
    _steger_check(ctx, N.STEGER_FAST, gray, 0.5, what="grating")


# ---- median / speckles -----------------------------------------------------------------------------------------------
def _speckle_ref(d, new_val, max_size, max_diff):
    e = d.copy()
    cv2.filterSpeckles(e, new_val, max_size, max_diff)
    return e


def test_median_tiny_shapes_and_extremes(ctx):
    rng = np.random.default_rng(2)
    for H, W in ((1, 1), (1, 2), (2, 1), (2, 2), (1, 301), (301, 1), (3, 1), (1, 3)):
        for d in (rng.integers(-40, 40, (H, W)), rng.choice([-32768, 32767, 0, -1], (H, W))):
            d = d.astype(np.int16)
            eq(ctx.median3_s16(d), cv2.medianBlur(d, 3), "median %dx%d" % (H, W))
    d = np.tile(np.array([[-32768, 32767], [32767, -32768]], np.int16), (20, 33))
    eq(ctx.median3_s16(d), cv2.medianBlur(d, 3), "median checkerboard of extremes")


def test_speckles_parameter_edges(ctx):
    rng = np.random.default_rng(3)
    shapes = ((1, 1), (1, 257), (257, 1), (2, 2), (40, 61))
    for H, W in shapes:
        d = (rng.integers(0, 6, (H, W)) * 16).astype(np.int16)
        d[rng.random((H, W)) < 0.2] = -16
        common = int(np.bincount((d.ravel().astype(np.int64) + 16)).argmax() - 16)
        for new_val in (-16, common):
            for max_size in (0, 1, 2, 25):
                for max_diff in (0, -1, 16, 32):
                    eq(ctx.filter_speckles(d, new_val, max_size, max_diff), _speckle_ref(d, new_val, max_size, max_diff),
                       "speckles %dx%d new %d size %d diff %d" % (H, W, new_val, max_size, max_diff))
    # maxDiff up to 32767 (cv2 4.13 narrows larger values to 16 bits: 65535 acts as -1 there, so they are not tested)
    d = np.tile(np.array([[-32768, 32767, 32767], [32767, -32768, -32768]], np.int16), (10, 10))
    for max_diff in (0, 1, 32766, 32767):
        eq(ctx.filter_speckles(d, 0, 3, max_diff), _speckle_ref(d, 0, 3, max_diff), "extremes diff %d" % max_diff)


def test_speckles_serpentine_component(ctx):
    """one single-pixel-wide path winding over a 720 x 1280 image (even rows full, odd rows one pixel at alternating
    ends), values rising and falling by 1 along it: one component of 461 159 pixels whose union-find chains run
    thousands of links deep.  maxSize one below its size keeps it, its size removes it."""
    H, W = 720, 1280
    path = []
    for y in range(0, H, 2):
        xs = range(W) if (y // 2) % 2 == 0 else range(W - 1, -1, -1)
        path += [(y, x) for x in xs]
        if y + 1 < H:
            path.append((y + 1, W - 1 if (y // 2) % 2 == 0 else 0))
    py, px = np.array(path).T
    tri = np.abs((np.arange(len(path)) % 200) - 100)  # steps of exactly 1 along the path
    d = np.full((H, W), -16, np.int16)
    d[py, px] = (tri * 3).astype(np.int16)
    size = len(path)
    for max_size, max_diff in ((size - 1, 3), (size, 3), (size - 1, 2)):
        want = _speckle_ref(d, -16, max_size, max_diff)
        eq(ctx.filter_speckles(d, -16, max_size, max_diff), want, "serpentine size %d diff %d" % (max_size, max_diff))
    assert (want != d).any() and (_speckle_ref(d, -16, size - 1, 3) == d).all()


# ---- disparity -> depth ----------------------------------------------------------------------------------------------
def _all_int16(seed):
    return np.random.default_rng(seed).permutation(np.arange(-32768, 32768)).astype(np.int16).reshape(256, 256)


def _q_matrices(golden_real):
    Qr = np.array([[1, 0, 0, -150.3], [0, 1, 0, -99.7], [0.001, 0.002, 0.0003, 233.123], [0.0001, 0.0002, 16.3, -0.7]])
    Qz = np.array([[1, 0, 0, -100.0], [0, 1, 0, -128.0], [1.0, 0, 0, -100.0], [1.0, 0, 0, -100.0]])  # 0/0 at x = 100
    Qi = np.array([[1, 0, 0, -100.0], [0, 1, 0, -128.0], [0, 0, 0, 300.0], [0, 1.0, 0, -77.0]])  # +-inf at y = 77
    return {"real": golden_real["Q"], "random": Qr, "zero_w_nan": Qz, "zero_w_inf": Qi}


def test_depth_every_int16_value(ctx, golden_real):
    """every int16 disparity at least once, through the rig's Q, a random Q with non-zero Q[3,3] and Q[2,0:2], two Qs
    whose W row is exactly zero at some pixels (0/0 -> NaN kept as in the reference, +-inf -> 0), and the default
    baseline"""
    for k, Q in _q_matrices(golden_real).items():
        for seed in (0, 1):
            d = _all_int16(seed)
            want = ref_ops.depth_from_disparity(d, Q)
            eq(ctx.disp_to_depth(d, Q), want, "depth Q %s" % k)
            if k == "zero_w_nan":
                assert np.isnan(want).any()
    for seed in (0, 1):
        d = _all_int16(seed)
        eq(ctx.disp_to_depth(d, None), ref_ops.depth_from_disparity(d, None), "depth default")


@pytest.mark.parametrize("use_wls", [True, False])
@pytest.mark.parametrize("qk", ["real", "zero_w_nan", None])
def test_depth_through_compute_depth(ctx, golden_real, use_wls, qk):
    """the fused depth in the WLS finalize kernel (with Q, default baseline) and the separate depth kernels: the depth
    plane equals depth_from_disparity of the disparity plane returned with it"""
    W, H, D, bs = 320, 360, 64, 5
    Q = _q_matrices(golden_real)[qk] if qk else None
    left, right = synth.stereo_pair(W, H, D, 6)
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    ctx.set_rectify_maps(0, maps[0], maps[1])
    ctx.set_rectify_maps(1, maps[2], maps[3])
    _, depth, disp = ctx.compute_depth(pipeline.depth_config(D, bs, 2, Q, use_wls=use_wls), left, right, want_disp=True)
    eq(depth, ref_ops.depth_from_disparity(disp, Q), "compute_depth depth")


# ---- reconstruction --------------------------------------------------------------------------------------------------
def _disp_recon_params(kind, ir, window=3, min_disparity=1.0):
    p = N.ReconParams()
    p.kind = kind
    p.fx, p.baseline, p.cx, p.cy = ir.fx, ir.baseline, ir.cx, ir.cy
    p.min_disparity = min_disparity
    p.window = window
    return p


def _edge_points(W, H, hw):
    xs = [-0.5, -0.49, 0.5, 1.5, 2.5, 3.5, hw - 0.5, hw - 0.5 + 1e-9, hw + 0.5, W - hw - 0.5, W - hw - 1.5, W - 0.5,
          W - 1.5, W - 0.51, 17.5, 18.5, 17.49999, 18.50001]
    ys = [-0.5, 0.5, 1.5, hw - 0.5, hw + 0.5, H - hw - 0.5, H - hw - 1.5, H - 0.5, 9.5, 10.5]
    return [(x, y) for x in xs for y in ys]


def _window_map(rng, W, H, window, mind):
    """cells of value quantised to 1/16 (ties in the sort) mixed with NaN, +-inf and values below min_disparity; each
    window centre on a 12-pixel grid gets 0, 1, 2, 4, window^2 - 1 or window^2 valid cells"""
    disp = (rng.integers(int(mind * 16) + 1, 40 * 16, (H, W)) / 16.0).astype(np.float32)
    bad = np.array([np.nan, np.inf, -np.inf, mind - 1 / 16, 0.0, -3.0], np.float32)
    hw, n2 = window // 2, window * window
    centres = []
    k = 0
    for y in range(hw + 1, H - hw - 1, 12):
        for x in range(hw + 1, W - hw - 1, 12):
            nvalid = min((0, 1, 2, 4, n2 - 1, n2)[k % 6], n2)
            k += 1
            cells = rng.permutation(n2)
            win = disp[y - hw:y + hw + 1, x - hw:x + hw + 1].reshape(-1)
            win[cells[nvalid:]] = rng.choice(bad, n2 - nvalid)
            disp[y - hw:y + hw + 1, x - hw:x + hw + 1] = win.reshape(window, window)
            centres.append((x, y))
    return disp, centres


def _ref_rows(fn, pts):
    r = fn(pts)
    return np.asarray(r, np.float32).reshape(-1, 3)


@pytest.mark.parametrize("window", [1, 3, 5, 7, 9])
def test_disparity_recon_windows_and_rounding(ctx, window):
    """DISPARITY and DISPARITY_MEDIAN on constructed float maps, bit for bit: points on .5 ties of even and odd k, at the
    window's bounds (px == hw, px == W - hw - 1), at -0.5; windows with 0, 1, an even number and all cells valid.
    The reference's int(round(x)) raises on NaN / inf coordinates; the library drops those points."""
    W, H = 150, 90
    rng = np.random.default_rng(window)
    Q = synth.camera_model(W, H)[1]
    ir = ref_ops.ImprovedLaserReconstructorRef(Q)
    hw = window // 2
    for mind in (1.0, -2.0):
        disp, centres = _window_map(rng, W, H, window, mind)
        pts = _edge_points(W, H, hw) + [(x + o, y - o) for (x, y) in centres for o in (0.0, 0.5, -0.5)]
        pts = [tuple(map(float, p)) for p in pts]
        xy = np.array(pts, np.float64)
        for kind, fn in ((N.RECON_DISPARITY, lambda p: ir.reconstruct_from_disparity(p, disp, mind)),
                         (N.RECON_DISPARITY_MEDIAN, lambda p: ir.reconstruct_with_interpolation(p, disp, window, mind))):
            want = _ref_rows(fn, pts)
            got = ctx.reconstruct(_disp_recon_params(kind, ir, window, mind), xy, disp).astype(np.float32)
            eq(got, want, "kind %d window %d min %.0f" % (kind, window, mind))
            assert len(want) > 0
            bad = np.array([(np.nan, 20.0), (20.0, np.nan), (np.inf, 20.0), (-np.inf, 20.0), (20.0, np.inf)])
            mixed = np.concatenate([bad, xy, bad])
            got = ctx.reconstruct(_disp_recon_params(kind, ir, window, mind), mixed, disp).astype(np.float32)
            eq(got, want, "kind %d with non-finite points" % kind)


def test_disparity_recon_z_bounds(ctx):
    """disparities whose Z lands on either side of 0 and 10: Z = fx * baseline / d must pass 0 < Z < 10 in float64"""
    W, H = 64, 8
    Q = synth.camera_model(W, H)[1]
    ir = ref_ops.ImprovedLaserReconstructorRef(Q)
    fxb = ir.fx * ir.baseline
    d10 = np.float32(fxb / 10.0)
    vals = [d10, np.nextafter(d10, np.float32(0)), np.nextafter(d10, np.float32(1e9)), np.float32(3e38),
            np.float32(1e-30), np.float32(-1e-30), np.float32(0.0), np.float32(-0.0), np.float32(1.5), np.float32(-7.0)]
    disp = np.ones((H, W), np.float32)
    pts = []
    for i, v in enumerate(vals):
        disp[2:7, 3 + 5 * i:8 + 5 * i] = v
        pts.append((5.0 + 5 * i, 4.0))
    for mind in (1.0, -10.0):
        for kind, fn in ((N.RECON_DISPARITY, lambda p: ir.reconstruct_from_disparity(p, disp, mind)),
                         (N.RECON_DISPARITY_MEDIAN, lambda p: ir.reconstruct_with_interpolation(p, disp, 3, mind))):
            want = _ref_rows(fn, pts)
            eq(ctx.reconstruct(_disp_recon_params(kind, ir, 3, mind), np.array(pts), disp).astype(np.float32), want,
               "z bounds kind %d min %.0f" % (kind, mind))


def test_plane_and_depth_recon_edges(ctx, golden_synth):
    """PLANE (rtol 1e-9) with NaN / inf pixels, which the reference drops itself; DEPTH bit for bit with int()'s
    truncation at -0.5 and W - 0.5 and depth values around 0"""
    g = golden_synth
    K = g["K"]
    W, H = 120, 80
    pts = [(x, y) for x in (-0.5, -0.49, 0.0, 0.5, 59.5, 60.5, W - 1.0, W - 0.5, W - 0.01, W + 0.0)
           for y in (-0.5, 0.0, 0.5, 40.5, H - 0.5, H - 0.01)]
    rng = np.random.default_rng(8)
    depth = rng.uniform(100, 3000, (H, W)).astype(np.float32)
    depth[rng.random((H, W)) < 0.2] = 0.0
    depth[rng.random((H, W)) < 0.05] = -1.0
    depth[rng.random((H, W)) < 0.05] = np.float32(1e-45)
    depth[rng.random((H, W)) < 0.05] = np.nan
    for refr in (0, 1):
        p = N.ReconParams()
        p.K[:] = list(K.reshape(9))
        p.plane[:] = list(synth.LASER_PLANE)
        p.use_refraction = refr
        p.n_water = 1.33
        rec = ref_ops.ReconstructorRef(K, synth.LASER_PLANE, bool(refr))
        p.kind = N.RECON_PLANE
        nonfin = [(np.nan, 3.0), (3.0, np.nan), (np.inf, 3.0), (-np.inf, -np.inf)]
        allp = pts + nonfin
        want = np.asarray(rec.reconstruct_laser_line(allp), np.float64).reshape(-1, 3)
        got = ctx.reconstruct(p, np.array(allp))
        assert got.shape == want.shape and np.allclose(got, want, rtol=1e-9, atol=1e-12)
        p.kind = N.RECON_DEPTH
        want = np.asarray(rec.reconstruct_from_depth(pts, depth), np.float64).reshape(-1, 3)
        eq(ctx.reconstruct(p, np.array(pts), depth), want, "from depth")
        eq(ctx.reconstruct(p, np.array(pts + nonfin), depth), want, "from depth, non-finite points dropped")


def _laser_depth_map_ref(pts, disp, fx, baseline):
    """ImprovedLaserReconstructor.create_laser_depth_map (improved_reconstruction.py:154-186) restated: depth at the
    rounded pixel where the disparity is > 1 and not NaN and 0 < depth < 10, f64 arithmetic, stored as f32"""
    h, w = disp.shape
    out = np.zeros((h, w), np.float32)
    for x, y in pts:
        px, py = int(round(x)), int(round(y))
        if 0 <= px < w and 0 <= py < h:
            d = disp[py, px]
            if d > 1.0 and not np.isnan(d):
                z = (fx * baseline) / d
                if 0 < z < 10:
                    out[py, px] = z
    return out


def test_laser_depth_map_duplicates_and_ties(ctx):
    W, H = 80, 40
    Q = synth.camera_model(W, H)[1]
    ir = ref_ops.ImprovedLaserReconstructorRef(Q)
    rng = np.random.default_rng(10)
    disp = rng.uniform(0.5, 60, (H, W)).astype(np.float32)
    disp[rng.random((H, W)) < 0.1] = np.nan
    disp[rng.random((H, W)) < 0.05] = np.inf
    disp[0, :] = np.float32(ir.fx * ir.baseline / 10.0)
    pts = [(k + 0.5, j + 0.5) for k in range(-1, W + 1, 3) for j in range(-1, H + 1, 2)]
    pts += [(9.5, 3.0), (10.5, 3.0), (10.0, 3.0), (10.4, 2.6), (11.5, 3.49), (12.5, 3.5), (3.0, -0.5), (W - 0.5, 2.0)]
    pts += [(float(x), 0.0) for x in range(W)]
    want = _laser_depth_map_ref(pts, disp, ir.fx, ir.baseline)
    eq(ctx.laser_depth_map(pts, disp, ir.fx, ir.baseline), want, "laser depth map")
    assert (want > 0).sum() > 50


# ---- point-cloud sink ------------------------------------------------------------------------------------------------
def _unique_voxel_cloud(rng, nx, ny, nz, vs):
    ijk = np.stack(np.meshgrid(np.arange(nx), np.arange(ny), np.arange(nz), indexing="ij"), -1).reshape(-1, 3)
    ijk = ijk[rng.permutation(len(ijk))] - np.array([nx // 2, ny // 3, 5])
    pts = (ijk + rng.uniform(0.1, 0.9, ijk.shape)) * vs
    assert np.array_equal(np.floor(pts / vs).astype(np.int64), ijk), "a point left its voxel"
    return pts, ijk


def test_voxel_downsample_9m_points(ctx):
    """9 M points, one per 2 mm voxel, permuted: past the second level of the exclusive scan and with a 2^25-slot
    hash table.  The mean of one point is the point, so the output is the input in input order.  Then a few thousand
    voxels get 1-59 more points, placed anywhere in the input: their means are the input-order f64 sums / counts."""
    vs = 0.002
    rng = np.random.default_rng(12)
    pts, ijk = _unique_voxel_cloud(rng, 300, 300, 100, vs)
    assert np.array_equal(ctx.voxel_downsample(pts, vs), pts)
    pick = rng.choice(len(pts), 3000, replace=False)
    extra_n = rng.integers(1, 60, len(pick))
    vid = np.repeat(pick, extra_n)
    extra = (ijk[vid] + rng.uniform(0.1, 0.9, (len(vid), 3))) * vs
    allp = np.concatenate([pts, extra])
    allv = np.concatenate([np.arange(len(pts)), vid])
    order = rng.permutation(len(allp))
    allp, allv = allp[order], allv[order]
    first = np.full(len(pts), len(allp))
    np.minimum.at(first, allv, np.arange(len(allp)))
    vox_order = np.argsort(first, kind="stable")
    want = allp[first[vox_order]].copy()
    rank = np.empty(len(pts), np.int64)
    rank[vox_order] = np.arange(len(pts))
    members = np.argsort(allv, kind="stable")
    starts = np.searchsorted(allv[members], pick)
    for v, k, s0 in zip(pick, extra_n, starts):
        idx = members[s0:s0 + k + 1]  # the voxel's points in input order
        s = allp[idx[0]].copy()
        for i in idx[1:]:
            s = s + allp[i]
        want[rank[v]] = s / (k + 1)
    got = ctx.voxel_downsample(allp, vs)
    eq(got, want, "voxel means")


def test_outlier_removal_neighbour_count_edges(ctx):
    rng = np.random.default_rng(13)
    for k in (1, 5, 20, 63):
        for n in (k, k + 1, k + 2, 200):
            pts = rng.normal(0, 0.1, (n, 3))
            pts[rng.random(n) < 0.1] = pts[0]
            want = np.asarray(ref_ops.simple_outlier_removal(pts, k, 1.0)).reshape(-1, 3)
            got = ctx.statistical_outlier_removal(pts, k, 1.0)
            eq(got, want, "n %d k %d" % (n, k))
    with pytest.raises(N.L3DError):
        ctx.statistical_outlier_removal(rng.normal(0, 0.1, (100, 3)), 64, 1.0)


# ---- device packing --------------------------------------------------------------------------------------------------
def test_pack_points_dev_across_launch_groups(ctx):
    """130 small frames, some without a laser line (0 points), packed in launches of 64 frames: every frame's rows
    must follow the previous frames' rows across the group boundaries"""
    W, H, D, bs, nf = 96, 64, 16, 5, 130
    K, Q = synth.camera_model(W, H)
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    base = [synth.stereo_pair(W, H, D, seed=s) for s in range(6)]
    blank = {0, 1, 63, 64, 65, 100, 127, 128, 129} | set(range(30, 40))
    L = np.stack([np.full_like(base[0][0], 30) if i in blank else base[i % 6][0] for i in range(nf)])
    R = np.stack([np.full_like(base[0][1], 30) if i in blank else base[i % 6][1] for i in range(nf)])
    cfg = pipeline.make_pipeline_config(W, H, D, bs, 1, Q, K, lanes=2, max_points=2000)
    fp = pipeline.FramePipeline(cfg, maps=maps, ctx=ctx)
    try:
        counts = fp.run_host(L, R)
        assert all(counts[i] == 0 for i in blank) and sum(c > 0 for c in counts) >= 100
        ids = [1000 + 3 * i for i in range(nf)]
        nrows = int(np.sum(counts))
        buf = ctx.lib.l3d_dev_alloc(ctx.h, max(nrows, 1) * 32)
        try:
            assert fp.pack_points_dev(ids, buf) == nrows
            table = np.empty((nrows, 4), np.float64)
            ctx.check(ctx.lib.l3d_memcpy_d2h(ctx.h, table.ctypes.data, buf, table.nbytes), "d2h")
        finally:
            ctx.lib.l3d_dev_free(ctx.h, buf)
        off = 0
        for i in range(nf):
            xyz = fp.fetch(i)["points_3d"]
            assert len(xyz) == counts[i]
            rows = table[off:off + counts[i]]
            assert (rows[:, 0] == ids[i]).all() and np.array_equal(rows[:, 1:], np.asarray(xyz, np.float64)), i
            off += counts[i]
    finally:
        fp.close()
