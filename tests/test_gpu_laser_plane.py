"""l3d_fit_plane against its numpy restatement (oracle/plane_fit.py), fit_laser_plane's refusals, and
LaserReconstructionSystem.calibrate_laser_plane end to end on a synthetic recording with a known laser plane."""
import ctypes as C
import json

import numpy as np
import pytest

import laser_3d_reconstruction_b200 as l3d
from laser_3d_reconstruction_b200 import _native as N
from laser_3d_reconstruction_b200 import pipeline, synth
from laser_3d_reconstruction_b200.improved_reconstruction import ImprovedLaserReconstructor
from oracle import plane_fit as opf

pytestmark = pytest.mark.gpu


def raw_fit(ctx, pts, threshold, hypotheses, seed):
    """l3d_fit_plane as called: -> (status, result struct, mask).  The result's hypothesis fields are filled even when the
    refinement is refused afterwards."""
    pts = np.ascontiguousarray(pts, np.float64).reshape(-1, 3)
    p = N.PlaneFitParams(float(threshold), int(hypotheses), int(seed))
    r = N.PlaneFitResult()
    mask = np.zeros(len(pts), np.uint8)
    rc = ctx.lib.l3d_fit_plane(ctx.h, N._ptr(pts), len(pts), C.byref(p), C.byref(r), N._ptr(mask))
    return rc, r, mask.astype(bool)


def plane_cloud(n, outliers, sigma, seed, plane=(0.3, -0.2, 0.9, 0.7)):
    """n points on `plane` (normalised) in a 1 m square, with Gaussian noise sigma along the normal; the first
    outliers * n replaced by uniform points in a 2 m cube"""
    rng = np.random.default_rng(seed)
    pl = np.asarray(plane, np.float64)
    pl = pl / np.linalg.norm(pl[:3])
    a = np.cross(pl[:3], [1.0, 0, 0]); a /= np.linalg.norm(a)
    b = np.cross(pl[:3], a)
    uv = rng.uniform(-0.5, 0.5, (n, 2))
    pts = -pl[3] * pl[:3] + uv[:, :1] * a + uv[:, 1:] * b + sigma * rng.standard_normal((n, 1)) * pl[:3]
    k = int(round(outliers * n))
    pts[rng.permutation(n)[:k]] = rng.uniform(-1, 1, (k, 3)) + [0, 0, 1]
    return pts, pl


def check_winner(ctx, pts, threshold, hypotheses, seed):
    rc, r, _ = raw_fit(ctx, pts, threshold, hypotheses, seed)
    try:
        win, cnt, _ = opf.ransac(pts, threshold, hypotheses, seed)
    except ValueError:  # no valid hypothesis: refused
        assert rc == -1
        return
    assert rc in (0, -1)  # -1: the refinement was left with fewer than 3 inliers
    assert (r.hypothesis, r.hypothesis_inliers) == (win, cnt)


# ---- 1. RANSAC winner, bit-exact ------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [3, 7, 1000, 200003])
@pytest.mark.parametrize("outliers", [0.0, 0.3, 0.7])
def test_winner_matches_oracle(ctx, n, outliers):
    for seed in ((0, 1, 0xDEADBEEFCAFEF00D) if n < 200003 else (5,)):
        pts, _ = plane_cloud(n, outliers, 2e-4, seed + n)
        for hyps in ((1, 64, 1024) if n < 200003 else (1, 64, 1024 if outliers == 0.3 else 64)):
            check_winner(ctx, pts, 1e-3, hyps, seed)


def test_winner_ties_boundaries_and_non_finite_points(ctx):
    rng = np.random.default_rng(11)
    # quantised clouds: every point of an integer grid, repeated and shuffled; the grid's symmetric planes tie
    for q, reps in ((3, 2), (4, 30), (6, 90)):
        g = np.stack(np.meshgrid(*[np.arange(q)] * 3, indexing="ij"), -1).reshape(-1, 3).astype(np.float64)
        pts = rng.permutation(np.tile(g, (reps, 1)))
        n = len(pts)
        for hyps in (1, 64, 1024):
            check_winner(ctx, pts, 0.5, hyps, n + hyps)
        _, cnt, counts = opf.ransac(pts, 0.5, 1024, n + 1024)
        assert (counts == cnt).sum() > 1  # ties for the most inliers really occur
    # points exactly at +-threshold of z = 0 (threshold 0.25) are inliers of every hypothesis through three z = 0 points
    xy = rng.integers(-20, 20, (3000, 2)).astype(np.float64)
    z = rng.choice([-0.25, 0.0, 0.25, 3.0], 3000)
    pts = np.c_[xy, z]
    for hyps in (64, 1024):
        check_winner(ctx, pts, 0.25, hyps, 3)
    win, cnt, _ = opf.ransac(pts, 0.25, 1024, 3)
    assert np.array_equal(np.abs(opf.hypothesis_planes(pts, 1024, 3)[0][win]), [0.0, 0.0, 1.0, 0.0])
    assert cnt == (np.abs(z) <= 0.25).sum()
    # NaN and inf points: never inliers, and a hypothesis that draws one is invalid
    pts, _ = plane_cloud(5000, 0.3, 2e-4, 4)
    bad = rng.permutation(5000)[:600]
    pts[bad[:200], 0] = np.nan
    pts[bad[200:400], 1] = np.inf
    pts[bad[400:], 2] = -np.inf
    for hyps in (1, 64, 1024):
        for seed in (0, 9):
            check_winner(ctx, pts, 1e-3, hyps, seed)
    rc, r, mask = raw_fit(ctx, pts, 1e-3, 1024, 0)
    assert rc == 0 and not mask[bad].any()


# ---- 2. refinement against float64 ----------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_refinement_matches_float64(ctx, seed):
    pts, _ = plane_cloud(20000 + 777 * seed, 0.4, 5e-4, 100 + seed)
    got = ctx.fit_plane(pts, 2e-3, 256, seed)
    want = opf.fit_plane(pts, 2e-3, 256, seed)
    assert (got["hypothesis"], got["hypothesis_inliers"]) == (want["hypothesis"], want["hypothesis_inliers"])
    assert np.abs(got["plane"] - want["plane"]).max() < 1e-9
    assert abs(got["rms"] - want["rms"]) < 1e-9 and np.abs(got["eig"] - want["eig"]).max() < 1e-9
    assert got["refits"] == want["refits"] and got["inliers"] == want["inliers"]
    assert np.array_equal(got["inlier_mask"], opf.inliers(pts, got["plane"], 2e-3))
    assert got["inliers"] == got["inlier_mask"].sum()


# ---- 3. recovery ----------------------------------------------------------------------------------------------------
def test_recovery(ctx):
    pts, pl = plane_cloud(10000, 0.4, 0.0, 21)
    got = ctx.fit_plane(pts, 1e-3, 1024, 0)
    assert np.abs(got["plane"][:3] - pl[:3]).max() < 1e-12 and abs(got["plane"][3] - pl[3]) < 1e-12
    pts, pl = plane_cloud(200000, 0.4, 3e-4, 22)
    fits = [ctx.fit_plane(pts, 1e-3, 1024, s) for s in (0, 0, 77)]
    a, b, c = fits
    ang = np.degrees(np.arccos(min(1.0, a["plane"][:3] @ pl[:3])))
    assert ang < 0.05 and abs(a["plane"][3] - pl[3]) < 1e-4
    for k in a:
        assert np.asarray(a[k]).tobytes() == np.asarray(b[k]).tobytes(), k  # two runs: identical bits
    assert np.abs(c["plane"] - a["plane"]).max() < 1e-9
    fit = l3d.fit_laser_plane(pts, threshold=1e-3)
    assert np.array_equal(fit.plane, ctx.fit_plane(pts, 1e-3, 1024, 0)["plane"]) and fit.inlier_mask.dtype == bool
    assert fit.spread > 0.5 and fit.inliers == fit.inlier_mask.sum()


# ---- 4. refusals ----------------------------------------------------------------------------------------------------
def test_refusals(ctx):
    pts, _ = plane_cloud(1000, 0.3, 2e-4, 5)
    for args in ((pts[:2], 1e-3, 64, 0), (pts, 0.0, 64, 0), (pts, -1e-3, 64, 0), (pts, np.nan, 64, 0), (pts, np.inf, 64, 0),
                 (pts, 1e-3, 0, 0), (pts, 1e-3, (1 << 20) + 1, 0), (pts, 1e-3, -5, 0)):
        with pytest.raises(N.L3DError, match="invalid argument"):
            ctx.fit_plane(*args)
    assert ctx.fit_plane(pts, 1e-3, 1 << 20, 0)["inliers"] > 600  # the largest hypothesis count is accepted
    with pytest.raises(N.L3DError, match="no hypothesis"):
        ctx.fit_plane(np.ones((100, 3)), 1e-3, 64, 0)  # every triple degenerate
    with pytest.raises(N.L3DError, match="no hypothesis"):
        ctx.fit_plane(np.full((100, 3), np.nan), 1e-3, 64, 0)
    with pytest.raises(N.L3DError, match="inlier"):
        ctx.fit_plane(np.random.default_rng(0).random((100, 3)), 1e-300, 1, 0)  # only p0 of the triple lies within
    assert ctx.fit_plane(pts, 1e-3, 64, 0)["inliers"] > 600  # the refusals left the context usable
    rng = np.random.default_rng(1)
    t = rng.uniform(0, 1, 5000)
    line = np.c_[0.1 + 0.2 * t, -0.1 + 0.05 * t, 0.5 + 0.3 * t] + 1e-6 * rng.standard_normal((5000, 3))
    with pytest.raises(ValueError, match="collinear"):
        l3d.fit_laser_plane(line, threshold=1e-4)
    uv = rng.uniform(-1, 1, (5000, 2))
    through_origin = np.c_[uv[:, 0], uv[:, 1], 0.5 * uv[:, 0] - 0.2 * uv[:, 1]]
    with pytest.raises(ValueError, match="optical centre"):
        l3d.fit_laser_plane(through_origin, threshold=1e-3)


# ---- 5. end to end on a synthetic recording -------------------------------------------------------------------------
W, H, D = 320, 360, 64


def true_plane():
    """the prototype's plane: tilted about both axes, crossing the stripe region at 0.38 .. 2.2 m"""
    f, B = 0.8 * W, 0.06
    Z0 = f * B / (0.35 * D)
    X0 = 0.05 * Z0
    pl = np.array([1.0, -0.1, 0.5, -(X0 + 0.5 * Z0)])
    pl = pl / np.linalg.norm(pl[:3])
    return -pl  # d >= 0, as the fit reports it


def recording(n=12):
    pl = true_plane()
    f, B = 0.8 * W, 0.06
    Ls, Rs, truth2, truth3 = [], [], [], []
    for k in range(n):
        scale = 0.75 + 0.5 * k / (n - 1)
        L, R, c = synth.plane_stripe_pair(W, H, D, pl, scale, seed=k)
        Ls.append(L); Rs.append(R)
        ok = ~np.isnan(c)
        y, x = np.arange(H, dtype=np.float64)[ok], c[ok]
        Z = f * B / (scale * (0.35 * D + 0.20 * D * np.sin(6 * x / W) * np.cos(4 * y / H)))
        truth2.append(np.c_[x, y]); truth3.append(np.c_[(x - W / 2) * Z / f, (y - H / 2) * Z / f, Z])
    return np.stack(Ls), np.stack(Rs), np.concatenate(truth2), np.concatenate(truth3), pl


def calibration_file(tmp_path):
    K, _ = synth.camera_model(W, H)
    calib = dict(R=np.eye(3).tolist(), T=[[-0.06], [0.0], [0.0]], camera_matrix_left=K.tolist(), dist_coeffs_left=[[0.0] * 5],
                 camera_matrix_right=K.tolist(), dist_coeffs_right=[[0.0] * 5])
    path = tmp_path / "stereo_calibration.json"
    path.write_text(json.dumps(calib))
    return str(path)


def make_system(path, use_wls):
    cam = l3d.SingleUSBStereoCameraManager(width=2 * W, height=H, split_mode='horizontal', calibration_file=path,
                                           use_wls=use_wls, verbose=False)
    assert cam.initialize_offline() and cam.Q is not None
    s = l3d.LaserReconstructionSystem(l3d.Config(), verbose=False)
    assert s.initialize(camera=cam)
    return s


@pytest.fixture(scope="module")
def rec():
    return recording()


@pytest.mark.parametrize("use_wls", [True, False])
def test_calibrate_laser_plane_end_to_end(tmp_path, rec, use_wls):
    """12 frames, Simple extractor, 1024 hypotheses, window 3.  The bounds are about twice the CPU prototype's (no WLS,
    true centres).  Measured on one NVIDIA B200 (1000 W):
    WLS off, threshold 5 mm (default):   4291 points, 3595 inliers, rms 2.47 mm, normal 0.280 deg, offset at the
                                         centroid 0.37 mm, relative 3D error median 0.35 % (p99 1.49 %).
    WLS on, threshold 10 mm (default):   4291 points, 3673 inliers, rms 4.3 mm, normal 0.191 deg, offset at the
                                         centroid 0.64 mm, relative 3D error median 0.11 % (p99 2.02 %).
    WLS on with 5 mm instead:            2653 inliers, 0.486 deg, 0.71 mm, 0.65 % -- outside the bounds.
    Why WLS wants the wider threshold: at the stripe the filtered disparity is noisier (10th-90th percentile of its error
    -0.47 .. +0.55 px against -0.30 .. +0.33 px without the filter, CPU restatement, true centres) and follows the
    field's curvature (error ~ 18 px^2 x Laplacian, 5 without).  Beyond ~1 m that is more than 5 mm of depth noise, so
    a 5 mm threshold keeps the near frames and only those far points that err towards the current plane; the
    selection tilts the normal.  The CPU restatement shows the same tilt (0.45 deg at 5 mm, 0.20 deg at 10 mm,
    0.05 deg at 20 mm), so it is the data, not the fit."""
    L, R, xy_true, p_true, pl_true = rec
    path = calibration_file(tmp_path)
    s = make_system(path, use_wls)
    caps = np.ascontiguousarray(np.concatenate([L, R], axis=2))
    fit = s.calibrate_laser_plane(frames=caps, lanes=3)  # default threshold: 10 mm with WLS, 5 mm without
    fit_views = s.calibrate_laser_plane(lefts=L, rights=R, lanes=5)
    for k in fit._fields:
        assert np.asarray(getattr(fit, k)).tobytes() == np.asarray(getattr(fit_views, k)).tobytes(), k
    # the fitted points are exactly the pipeline's per-frame DISPARITY_MEDIAN points
    cam = s.camera
    recon = ImprovedLaserReconstructor(cam.Q, verbose=False).recon_params(N.RECON_DISPARITY_MEDIAN, 1.0, 3)
    ex = s.laser_extractor
    pc = pipeline.make_pipeline_config(W, H, 64, 5, 2, None, s.reconstructor.K, extractor=N.EXTRACT_SIMPLE, lanes=2,
                                       max_points=20000, bright_thr=int(ex.brightness_threshold),
                                       hsv_lo=tuple(int(v) for v in ex.hsv_lower), hsv_hi=tuple(int(v) for v in ex.hsv_upper),
                                       min_area=float(ex.min_area), recon=recon)
    pc.depth = cam._depth_config()
    fp = pipeline.FramePipeline(pc, maps=(cam.map_left_x, cam.map_left_y, cam.map_right_x, cam.map_right_y))
    try:
        counts = fp.run_host(np.ascontiguousarray(L), np.ascontiguousarray(R))
    finally:
        fp.close()
    assert len(fit.inlier_mask) == counts.sum() > 3000
    # accuracy against the rendered plane
    ang = np.degrees(np.arccos(min(1.0, abs(fit.plane[:3] @ pl_true[:3]))))
    c = p_true.mean(0)
    offset = abs(fit.plane[:3] @ c + fit.plane[3])
    p_hat = l3d.Reconstructor(s.reconstructor.K, fit.plane, use_refraction_correction=False).reconstruct_laser_line(xy_true)
    rel = np.linalg.norm(p_hat - p_true, axis=1) / p_true[:, 2]
    print("\nplane fit (WLS %s): %d points, %d inliers, rms %.3g mm, spread %.3f, normal error %.4f deg, offset at the "
          "centroid %.4f mm, relative 3D error median %.4f %% p99 %.4f %%" % (
              "on" if use_wls else "off", len(fit.inlier_mask), fit.inliers, 1e3 * fit.rms, fit.spread, ang, 1e3 * offset,
              100 * np.median(rel), 100 * np.percentile(rel, 99)))
    assert ang <= 0.5 and offset <= 1e-3 and np.median(rel) <= 5e-3
    assert np.array_equal(s.reconstructor.laser_plane, fit.plane)
    assert np.array_equal(s.config.LASER_PLANE_COEFFICIENTS, fit.plane)
    assert np.array_equal(l3d.Config.LASER_PLANE_COEFFICIENTS, [0, 0, 1, 0])
    assert s.point_cloud == [] and s.frame_count == 0
    # process_frames afterwards gives exactly what a fresh system gives
    out = s.process_frames(frames=caps, lanes=3)
    fresh = make_system(path, use_wls)
    want = fresh.process_frames(frames=caps, lanes=3)
    assert len(out) == len(want) == len(L)
    for (a_rect, a_depth, a_pts), (b_rect, b_depth, b_pts) in zip(out, want):
        assert np.array_equal(a_rect, b_rect) and a_depth.tobytes() == b_depth.tobytes() and a_pts == b_pts
    assert s.point_cloud == fresh.point_cloud and s.frame_count == fresh.frame_count == len(L)
    s.stop(); fresh.stop()
