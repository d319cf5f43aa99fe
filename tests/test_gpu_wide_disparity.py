"""StereoSGBM with numDisparities in (256, 512]: 16 disparities per lane, 9-bit disparity index in the winner-takes-all
keys, SGBM_3WAY's arg-min with two slots of every d mod 8 class per lane.  Every matcher output is bit-exact against
cv2 and, for the volumes, against the oracle's C restatement; the depth path and the frame pipeline against the
stage-wise reference path.

The scenes are built here: synth.stereo_pair spans 0.15 D .. 0.55 D and never reaches a disparity index above 255.
Every case asserts that a stated share of cv2's valid pixels has an index (disparity - minDisparity) of at least 256,
so that no equality holds because the wide indices never occur."""
import cv2
import numpy as np
import pytest

from laser_3d_reconstruction_b200 import _native as N
from laser_3d_reconstruction_b200 import pipeline, stereo, synth
from oracle import cref, ref_ops

pytestmark = pytest.mark.gpu


def eq(a, b, what=""):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, "%s: shape %s vs %s" % (what, a.shape, b.shape)
    bad = np.argwhere(a != b)
    assert len(bad) == 0, "%s: %d/%d differ, first %s got %s want %s" % (
        what, len(bad), a.size, tuple(bad[0]), a[tuple(bad[0])], b[tuple(bad[0])])


def band_levels(W, D, role, rng):
    """Integer disparity of each 40-column band (indexed by the right view's column, as in synth.stereo_pair).
    "left": levels for a matcher with minDisparity 0, in [max(D - 96, 160), D - 6], every second band at 262 or more;
    "right": levels for the right matcher (minDisparity = -(D - 1), views swapped, index = D - 1 - disparity), in
    [2, 90], every second band at D - 260 or less;  "both": right levels on the left half of the image, where the right
    matcher's valid columns are, left levels on the right half.  Neighbouring bands differ by at most 96 pixels except
    at the middle of a "both" scene."""
    nb = W // 40 + 1
    out = np.empty(nb, np.int64)
    for k in range(nb):
        kind = role if role != "both" else ("left" if (k + 0.5) * 40 >= W / 2 else "right")
        if kind == "left":
            lo, hi = max(D - 96, 160), D - 6
            out[k] = rng.integers(max(lo, 262) if k % 2 else lo, hi + 1)
        else:
            hi = 90
            out[k] = rng.integers(2, (min(D - 260, hi) if k % 2 else hi) + 1)
    return out


def wide_pair(W, H, D, seed, role="both", laser=False):
    """(left, right) BGR uint8: blurred noise texture seen through fronto-parallel bands (band_levels), optionally with
    the green laser stripe the extractors look for."""
    rng = np.random.default_rng(seed)
    pad = D + 16
    tex = rng.integers(0, 256, (H, W + 2 * pad, 3)).astype(np.float32)
    tex = np.clip((cv2.GaussianBlur(tex, (0, 0), 1.5) - 128.0) * 2.2 + 110.0, 0, 200)
    levels = band_levels(W, D, role, rng)
    d = np.broadcast_to(levels[np.arange(W) // 40][None, :], (H, W))
    xs = np.arange(W)[None, :]
    ys = np.arange(H)[:, None]
    left = tex[ys, xs + pad]
    right = tex[ys, xs + pad + d]
    if laser:
        colour = np.array([140.0, 255.0, 140.0], np.float32)
        cx = 0.7 * W + 0.05 * W * np.sin(5 * np.arange(H) / H)
        a = np.clip(3.0 * np.exp(-(xs - cx[:, None]) ** 2 / (2 * 2.5 ** 2)), 0, 1)[..., None]
        left = left * (1 - a) + colour * a
        dc = d[np.arange(H), np.clip(np.rint(cx).astype(int), 0, W - 1)]
        a = np.clip(3.0 * np.exp(-(xs - (cx - dc)[:, None]) ** 2 / (2 * 2.5 ** 2)), 0, 1)[..., None]
        right = right * (1 - a) + colour * a
    return np.rint(left).astype(np.uint8), np.rint(right).astype(np.uint8)


def gray(img):
    return cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)


def wide_share(disp16, minD):
    """share of the valid pixels of a matcher output whose disparity index d - minDisparity is at least 256"""
    valid = disp16 != (minD - 1) * 16
    if not valid.any():
        return 0.0
    return float((disp16[valid].astype(np.int32) - 16 * minD >= 256 * 16).mean())


SHARE = 0.2  # stated share of cv2's valid pixels with a disparity index >= 256, per matcher output


@pytest.mark.parametrize("mode", [0, 1, 2, 3])
@pytest.mark.parametrize("bs", [5, 7, 11])
@pytest.mark.parametrize("D", [272, 320, 384, 512])
def test_wide_sgbm_all_roles(ctx, D, bs, mode):
    """The as-constructed matcher (uniquenessRatio 10, speckle filter), the WLS-mutated one and the right matcher: C and S
    against the oracle (modes SGBM / HH / HH4), the raw disparity against the oracle, the final disparity against cv2,
    and the production call (WTA fused into the last path, no S written) against cv2."""
    W, H = D + 224, 40 + 4 * (bs % 4)
    base, mut, right = ref_ops.sgbm_param_sets(D, bs, mode)
    for role, kw in (("base", base), ("mutated", mut), ("right", right)):
        lb, rb = wide_pair(W, H, D, D + bs + 10 * mode, role="right" if role == "right" else "left")
        lg, rg = gray(lb), gray(rb)
        if role == "right":
            lg, rg = rg, lg
        tag = "D%d bs%d m%d %s" % (D, bs, mode, role)
        want = cv2.StereoSGBM_create(**kw).compute(lg, rg)
        share = wide_share(want, kw["minDisparity"])
        assert share >= SHARE, "%s: only %.3f of cv2's valid pixels have a disparity index >= 256" % (tag, share)
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
        eq(ctx.sgbm_compute(p, lg, rg), want, tag + " fused-WTA disp vs cv2")


@pytest.mark.parametrize("H", [5, 8, 12, 20, 28])
def test_wide_sgbm_3way_few_rows(ctx, H):
    """SGBM_3WAY at D = 320 on images of a few rows: OpenCV's shifted stripe rows together with the 16-disparities-per-lane
    arg-min, with and without the uniqueness test."""
    D, W = 320, 560
    lb, rb = wide_pair(W, H, D, H, role="left")
    lg, rg = gray(lb), gray(rb)
    for bs in (5, 11):
        for (uq, d12, sw) in ((0, 5, 0), (10, 1, 0), (0, 1000000, 20)):
            kw = dict(minDisparity=0, numDisparities=D, blockSize=bs, P1=24 * bs * bs, P2=96 * bs * bs, disp12MaxDiff=d12,
                      preFilterCap=63, uniquenessRatio=uq, speckleWindowSize=sw, speckleRange=2, mode=2)
            want = cv2.StereoSGBM_create(**kw).compute(lg, rg)
            tag = "3way H%d bs%d u%d" % (H, bs, uq)
            assert wide_share(want, 0) >= SHARE, tag
            p = N.SgbmParams(**kw)
            eq(ctx.sgbm_compute(p, lg, rg), want, tag)
            disp, raw = ctx.sgbm_compute(p, lg, rg, want_raw=True)
            eq(disp, want, tag + " (raw read back)")
            eq(raw, cref.sgbm_compute(lg, rg, want_raw=True, **kw)[1], tag + " raw vs oracle")


@pytest.mark.parametrize("mode", [1, 0, 3, 2])
@pytest.mark.parametrize("D", [320, 384])
def test_wide_sgbm_pair(ctx, D, mode):
    """The matcher pair of one frame in one call (two single cost passes at these geometries): both disparities equal
    cv2's, both cost volumes equal the single-matcher path's."""
    W, H, bs = D + 400, 48, 7
    lb, rb = wide_pair(W, H, D, D + mode)
    lg, rg = gray(lb), gray(rb)
    _, mut, right = ref_ops.sgbm_param_sets(D, bs, mode)
    pl, pr = N.SgbmParams(**mut), N.SgbmParams(**right)
    want_l = cv2.StereoSGBM_create(**mut).compute(lg, rg)
    want_r = cv2.StereoSGBM_create(**right).compute(rg, lg)
    assert wide_share(want_l, 0) >= SHARE and wide_share(want_r, -(D - 1)) >= SHARE
    dl, dr, Cl, Cr = ctx.sgbm_compute_pair(pl, pr, lg, rg, want_volumes=True)  # SGBM_3WAY: its striped volumes
    eq(Cl, ctx.sgbm_compute(pl, lg, rg, want_volumes=True)[1], "D%d m%d left cost volume" % (D, mode))
    eq(Cr, ctx.sgbm_compute(pr, rg, lg, want_volumes=True)[1], "D%d m%d right cost volume" % (D, mode))
    eq(dl, want_l, "D%d m%d left disparity vs cv2" % (D, mode))
    eq(dr, want_r, "D%d m%d right disparity vs cv2" % (D, mode))


def test_wide_stereo_classes(ctx):
    """The cv2 look-alike classes pass numDisparities through: StereoSGBM at 320 and its right matcher equal cv2."""
    D = 320
    lb, rb = wide_pair(D + 400, 48, D, 3)
    lg, rg = gray(lb), gray(rb)
    kw = dict(minDisparity=0, numDisparities=D, blockSize=7, P1=24 * 49, P2=96 * 49, disp12MaxDiff=1, uniquenessRatio=10,
              speckleWindowSize=100, speckleRange=32, preFilterCap=63, mode=1)
    m = stereo.StereoSGBM_create(**kw)
    want = cv2.StereoSGBM_create(**kw).compute(lg, rg)
    assert wide_share(want, 0) >= SHARE
    eq(m.compute(lg, rg), want, "StereoSGBM class")
    rm = stereo.createRightMatcher(m)
    rp = rm.params()
    want_r = cv2.StereoSGBM_create(**{f: getattr(rp, f) for f, _ in N.SgbmParams._fields_}).compute(rg, lg)
    assert rp.minDisparity == -(D - 1) and wide_share(want_r, -(D - 1)) >= SHARE
    eq(rm.compute(rg, lg), want_r, "right matcher class")


@pytest.mark.parametrize("mode,use_wls", [(1, True), (2, True), (1, False), (0, False)])
def test_wide_compute_depth(ctx, mode, use_wls):
    """get_frames()'s depth path at 960x270 / D 384: the rectified view exact, the matcher outputs exact against cv2, the
    filtered disparity within the depth tests' tolerance classes (WLS: <= 1 LSB on >= 99.9 % of the pixels, the depth
    exact where the disparity is), and the serial FGS solver bit-identical to the oracle."""
    W, H, D, bs = 960, 270, 384, 9
    left, right = wide_pair(W, H, D, 21 + mode, laser=True)
    K, Q = synth.camera_model(W, H)
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    ctx.set_rectify_maps(0, maps[0], maps[1])
    ctx.set_rectify_maps(1, maps[2], maps[3])
    dc = pipeline.depth_config(D, bs, mode, Q, use_wls=use_wls)
    rect, depth, disp = ctx.compute_depth(dc, left, right, want_disp=True)
    wrect, wdepth, aux = ref_ops.depth_path(left, right, maps, D, bs, mode, Q, use_wls=use_wls, want_all=True)
    eq(rect, wrect, "rectified left")
    assert wide_share(aux["dl"], 0) >= SHARE
    if use_wls:
        assert wide_share(aux["dr"], -(D - 1)) >= SHARE
        diff = np.abs(disp.astype(np.int32) - aux["df"].astype(np.int32))
        assert (diff <= 1).mean() >= 0.999, "wls: %.5f within 1 LSB" % (diff <= 1).mean()
        ok = diff == 0
        assert np.array_equal(depth[ok], wdepth[ok])
        # the two matchers feeding the filter, and the filter with the serial solver, bit for bit
        _, mut, right_kw = ref_ops.sgbm_param_sets(D, bs, mode)
        dl, dr = ctx.sgbm_compute_pair(N.SgbmParams(**mut), N.SgbmParams(**right_kw), aux["lg"], aux["rg"])
        eq(dl, aux["dl"], "left disparity vs cv2")
        eq(dr, aux["dr"], "right disparity vs cv2")
        r = int(np.ceil(0.5 * bs))
        got1 = ctx.wls_filter(N.WlsParams(8000.0, 1.5, 0, D, r, 24, N.WLS_SOLVER_SERIAL), dl, dr, aux["lg"])
        eq(got1, aux["df"], "serial FGS solver vs oracle")
    else:
        eq(disp, aux["df"], "disparity")
        eq(depth, wdepth, "depth")


def _run_pipeline(ctx, cfg, maps, L, R, frames):
    fp = pipeline.FramePipeline(cfg, maps=maps, ctx=ctx)
    try:
        fp.run_dev(fp.upload(L), fp.upload(R), len(L))
        return [fp.fetch(i) for i in frames]
    finally:
        fp.close()


@pytest.mark.parametrize("mode", [1, 2])
def test_wide_pipeline_lanes(ctx, mode):
    """The frame pipeline at 960x270 / D 384: two lanes and eight lanes (which ask for grouping: at D > 256 it falls back
    to lane-per-frame) give identical per-frame outputs, equal to the stage-by-stage compute_depth call."""
    W, H, D, bs = 960, 270, 384, 9
    K, Q = synth.camera_model(W, H)
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    pairs = [wide_pair(W, H, D, 30 + s, laser=True) for s in range(3)]
    idx = [0, 1, 2, 0, 1, 2, 0, 1, 2]
    L = np.stack([pairs[i][0] for i in idx])
    R = np.stack([pairs[i][1] for i in idx])
    results = {}
    for lanes in (2, 8):
        cfg = pipeline.make_pipeline_config(W, H, D, bs, mode, Q, K, extractor=N.STEGER_IMPROVED, lanes=lanes, max_points=8000)
        results[lanes] = _run_pipeline(ctx, cfg, maps, L, R, range(len(idx)))
    for i in range(len(idx)):
        for k in ("left_rect", "depth", "disp16", "points_2d", "points_3d"):
            eq(results[2][i][k], results[8][i][k], "lanes 2 vs 8 %s frame %d" % (k, i))
            eq(results[8][i][k], results[8][idx[i]][k], "same input in another lane %s frame %d" % (k, i))
    ctx.set_rectify_maps(0, maps[0], maps[1])
    ctx.set_rectify_maps(1, maps[2], maps[3])
    for s in range(3):
        rect, depth, disp = ctx.compute_depth(pipeline.depth_config(D, bs, mode, Q), pairs[s][0], pairs[s][1], want_disp=True)
        eq(results[8][s]["left_rect"], rect, "pipeline vs compute_depth rect frame %d" % s)
        eq(results[8][s]["disp16"], disp, "pipeline vs compute_depth disparity frame %d" % s)
        eq(results[8][s]["depth"], depth, "pipeline vs compute_depth depth frame %d" % s)
    assert len(results[8][0]["points_3d"]) > 0


def test_wide_pipeline_full_size(ctx):
    """One 1920x1080 frame at D 384 / block 11, MODE_HH through the frame pipeline: the matcher pair equals cv2 bit for bit,
    the filtered disparity is within the WLS tolerance of the stage-wise reference path, and the pipeline's frame equals
    the stage-by-stage compute_depth call."""
    W, H, D, bs, mode = 1920, 1080, 384, 11, 1
    K, Q = synth.camera_model(W, H)
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    left, right = wide_pair(W, H, D, 77, laser=True)
    cfg = pipeline.make_pipeline_config(W, H, D, bs, mode, Q, K, extractor=N.STEGER_IMPROVED, lanes=2, max_points=20000)
    got = _run_pipeline(ctx, cfg, maps, left[None], right[None], [0])[0]
    wrect, wdepth, aux = ref_ops.depth_path(left, right, maps, D, bs, mode, Q, want_all=True)
    eq(got["left_rect"], wrect, "rectified image vs cv2.remap")
    assert wide_share(aux["dl"], 0) >= SHARE and wide_share(aux["dr"], -(D - 1)) >= SHARE
    _, mut, right_kw = ref_ops.sgbm_param_sets(D, bs, mode)
    dl, dr = ctx.sgbm_compute_pair(N.SgbmParams(**mut), N.SgbmParams(**right_kw), aux["lg"], aux["rg"])
    eq(dl, aux["dl"], "left disparity vs cv2")
    eq(dr, aux["dr"], "right disparity vs cv2")
    diff = np.abs(got["disp16"].astype(np.int32) - aux["df"].astype(np.int32))
    assert (diff <= 1).mean() >= 0.999
    ctx.set_rectify_maps(0, maps[0], maps[1])
    ctx.set_rectify_maps(1, maps[2], maps[3])
    _, depth, disp = ctx.compute_depth(pipeline.depth_config(D, bs, mode, Q), left, right, want_disp=True)
    eq(got["disp16"], disp, "pipeline vs compute_depth disparity")
    eq(got["depth"], depth, "pipeline vs compute_depth depth")


def wide_kw(D, bs, mode=1):
    """the WLS-mutated matcher with penalties small enough for blocks up to 21 (P2 + bs^2 (2 ftzero + 63) < 2^16)"""
    return dict(ref_ops.sgbm_param_sets(D, bs, mode)[1], P1=2 * bs * bs, P2=8 * bs * bs, preFilterCap=15)


def test_wide_limits(ctx):
    """numDisparities above 512 keeps failing with L3D_ERR_UNSUPPORTED, naming the supported range, and so does a
    blockSize above 15 with more than 272 disparities (the cost kernel's tile); the context stays usable afterwards.
    The largest accepted blocks on both sides of that line (21 at D 272, 15 at D 288 and 512) equal cv2."""
    D = 512
    lb, rb = wide_pair(D + 200, 24, D, 5, role="left")
    lg, rg = gray(lb), gray(rb)
    for bad in (528, 1024):
        kw = dict(ref_ops.sgbm_param_sets(bad, 5, 1)[1])
        with pytest.raises(N.L3DError, match=r"\(-3\).*\[16,512\]"):  # L3D_ERR_UNSUPPORTED
            ctx.sgbm_compute(N.SgbmParams(**kw), lg, rg)
        with pytest.raises(N.L3DError, match=r"\(-3\).*\[16,512\]"):
            ctx.sgbm_compute_pair(N.SgbmParams(**kw), N.SgbmParams(**dict(kw, minDisparity=-(bad - 1))), lg, rg)
    for bad_D, bad_bs in ((288, 17), (320, 17), (384, 19), (512, 21)):
        kw = wide_kw(bad_D, bad_bs)
        with pytest.raises(N.L3DError, match=r"\(-3\).*blockSize <= 15 above 272"):
            ctx.sgbm_compute(N.SgbmParams(**kw), lg, rg)
        with pytest.raises(N.L3DError, match=r"\(-3\).*blockSize <= 15 above 272"):
            ctx.sgbm_compute_pair(N.SgbmParams(**kw), N.SgbmParams(**dict(kw, minDisparity=-(bad_D - 1))), lg, rg)
        with pytest.raises(N.L3DError):
            stereo.StereoSGBM_create(**kw).compute(lg, rg)
    for good_D, good_bs in ((272, 21), (288, 15), (512, 15)):
        kw = dict(wide_kw(good_D, good_bs), mode=0)
        lb2, rb2 = wide_pair(good_D + 224, 48, good_D, good_bs, role="left")
        lg2, rg2 = gray(lb2), gray(rb2)
        want = cv2.StereoSGBM_create(**kw).compute(lg2, rg2)
        assert wide_share(want, 0) >= SHARE, (good_D, good_bs)
        eq(ctx.sgbm_compute(N.SgbmParams(**kw), lg2, rg2), want, "D%d block %d vs cv2" % (good_D, good_bs))
    _, mut, _ = ref_ops.sgbm_param_sets(D, 5, 1)
    want = cv2.StereoSGBM_create(**mut).compute(lg, rg)
    assert wide_share(want, 0) >= SHARE
    eq(ctx.sgbm_compute(N.SgbmParams(**mut), lg, rg), want, "after the errors")
