"""Generate tests/golden/*.npz by running the REAL reference (imported from /root/reference) in the
build container.  The reference cannot travel to the GPU box, so its outputs are committed here as
small fixtures together with this script.

    python tests/golden/make_golden.py

Inputs are stored with the outputs so that nothing depends on re-generating them bit-identically.
"""
import contextlib
import io
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)

from laser_3d_reconstruction_b200 import synth  # noqa: E402


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def pts(a, dtype=np.float64):
    return np.array(a, dtype=dtype).reshape(-1, 2)


def main():
    from config import Config
    from core.laser_extractor import FastStegerExtractor, SimpleLaserExtractor
    from core.reconstruction import Reconstructor
    from improved_reconstruction import ImprovedLaserReconstructor
    from improved_steger import HybridLaserExtractor, ImprovedStegerExtractor
    from camera.single_usb_stereo_camera import SingleUSBStereoCameraManager

    # ---------------- synthetic c1 frame: extractors + reconstructors -----------------------
    W, H, D = 320, 360, 64
    left, right = synth.stereo_pair(W, H, D, seed=0)
    K, Q = synth.camera_model(W, H)
    out = dict(left=left, right=right, K=K, Q=Q, W=W, H=H, D=D)

    simple_cfg = quiet(SimpleLaserExtractor, hsv_lower=Config.SIMPLE_LASER_HSV_LOWER, hsv_upper=Config.SIMPLE_LASER_HSV_UPPER,
                       brightness_threshold=Config.SIMPLE_LASER_BRIGHTNESS_THRESHOLD, min_area=Config.SIMPLE_LASER_MIN_AREA)
    simple_def = quiet(SimpleLaserExtractor)
    out["simple_cfg"] = pts(quiet(simple_cfg.extract_centerline, left))
    out["simple_def"] = pts(quiet(simple_def.extract_centerline, left))
    fast = quiet(FastStegerExtractor, sigma=3.0, brightness_threshold=200)
    out["fast"] = pts(quiet(fast.extract_centerline, left), np.float32)
    out["fast_roi"] = pts(quiet(fast.extract_centerline, left, (100, 40, 150, 200)), np.float32)
    out["fast_gray"] = pts(quiet(fast.extract_centerline, cv2.cvtColor(left, cv2.COLOR_BGR2GRAY)), np.float32)
    imp = quiet(ImprovedStegerExtractor, sigma=3.0, brightness_threshold=200, response_threshold=0.5)
    out["improved"] = pts(quiet(imp.extract_centerline, left))
    out["optimized"] = pts(quiet(imp.extract_centerline_optimized, left))
    hyb = quiet(HybridLaserExtractor)
    out["hybrid"] = pts(quiet(hyb.extract_centerline, left))

    # depth map for reconstruct_from_depth: the get_frames() arithmetic with the real cv2 matcher
    lg, rg = cv2.cvtColor(left, cv2.COLOR_BGR2GRAY), cv2.cvtColor(right, cv2.COLOR_BGR2GRAY)
    m = cv2.StereoSGBM_create(minDisparity=0, numDisparities=D, blockSize=5, P1=600, P2=2400, disp12MaxDiff=1,
                              uniquenessRatio=10, speckleWindowSize=100, speckleRange=32, preFilterCap=63,
                              mode=cv2.STEREO_SGBM_MODE_SGBM_3WAY)
    disp16 = m.compute(lg, rg)
    disp = disp16.astype(np.float32) / 16.0
    depth = cv2.reprojectImageTo3D(disp, Q)[:, :, 2]
    with np.errstate(invalid="ignore"):
        depth[depth < 0] = 0; depth[depth > 10] = 0; depth[disp <= 0] = 0
    out["disp16_3way"] = disp16
    out["depth"] = depth
    for name, refr in (("rec_air", False), ("rec_water", True)):
        rec = Reconstructor(K, synth.LASER_PLANE, use_refraction_correction=refr)
        simple_pts = [tuple(p) for p in out["simple_cfg"]]
        out[name + "_depth"] = np.asarray(rec.reconstruct_from_depth(simple_pts, depth), np.float64).reshape(-1, 3)
        out[name + "_line"] = np.asarray(rec.reconstruct_laser_line(simple_pts), np.float64).reshape(-1, 3)
    rec = Reconstructor(K, synth.LASER_PLANE, use_refraction_correction=True)
    fast_pts = quiet(fast.extract_centerline, left)
    out["rec_fast_depth"] = np.asarray(rec.reconstruct_from_depth(fast_pts, depth), np.float64).reshape(-1, 3)
    out["rec_fast_line"] = np.asarray(rec.reconstruct_laser_line(fast_pts), np.float64).reshape(-1, 3)
    irec = quiet(ImprovedLaserReconstructor, Q)
    ipts = [tuple(p) for p in out["optimized"]]
    out["irec_disp"] = np.asarray(quiet(irec.reconstruct_from_disparity, ipts, disp), np.float32).reshape(-1, 3)
    out["irec_interp"] = np.asarray(quiet(irec.reconstruct_with_interpolation, ipts, disp, 3, 1.0), np.float32).reshape(-1, 3)
    np.savez_compressed(os.path.join(HERE, "synth_c1.npz"), **out)

    # ---------------- real 320x240 pair + shipped calibration: camera class ------------------
    names = sorted(os.listdir(os.path.join(REF, "calibration_images", "left")))
    real = {}
    cam = quiet(SingleUSBStereoCameraManager, camera_id=0, width=640, height=240,
                calibration_file=os.path.join(REF, "stereo_calibration.json"))
    assert quiet(cam._load_calibration)
    try:
        quiet(cam._initialize_stereo_matcher_optimized)  # dies at cv2.ximgproc after creating stereo_matcher
    except AttributeError:
        pass
    assert cam.stereo_matcher is not None
    intr = cam.get_camera_intrinsics()
    real.update(K_left=cam.camera_matrix_left, dist_left=cam.dist_coeffs_left, K_right=cam.camera_matrix_right,
                dist_right=cam.dist_coeffs_right, R=cam.R, T=cam.T, Q=cam.Q, P1=cam.P1,
                intr=np.array([intr[k] for k in ("fx", "fy", "cx", "cy", "baseline")]),
                map_left_x=cam.map_left_x[::8, ::8].copy(), map_left_y=cam.map_left_y[::8, ::8].copy())
    for tag, idx in (("a", 0), ("b", 13)):
        l = cv2.imread(os.path.join(REF, "calibration_images", "left", names[idx]))
        r = cv2.imread(os.path.join(REF, "calibration_images", "right", names[idx].replace("left_", "right_")))
        combined = np.hstack([l, r])
        lv, rv = cam._split_frame(combined)
        lrect = cv2.remap(lv, cam.map_left_x, cam.map_left_y, cv2.INTER_LINEAR)
        rrect = cv2.remap(rv, cam.map_right_x, cam.map_right_y, cv2.INTER_LINEAR)
        lgray = cv2.cvtColor(lrect, cv2.COLOR_BGR2GRAY)
        rgray = cv2.cvtColor(rrect, cv2.COLOR_BGR2GRAY)
        d16 = cam.stereo_matcher.compute(lgray, rgray)  # as constructed: 3WAY, 64/5, uniq 10, speckle 100/32
        dispf = d16.astype(np.float32) / 16.0
        dep = cv2.reprojectImageTo3D(dispf, cam.Q)[:, :, 2]
        with np.errstate(invalid="ignore"):
            dep[dep < 0] = 0; dep[dep > 10] = 0; dep[dispf <= 0] = 0
        real.update({"frame_" + tag: combined, "lrect_" + tag: lrect, "rrect_" + tag: rrect, "disp16_" + tag: d16,
                     "depth_" + tag: dep})
    # one file per pair (and the calibration apart) keeps every golden file under 1 MB
    files = {"real_pair_" + t + ".npz": {k: v for k, v in real.items() if k.endswith("_" + t)} for t in ("a", "b")}
    files["real_rig.npz"] = {k: v for k, v in real.items() if not k.endswith(("_a", "_b"))}
    for f, arrays in files.items():
        np.savez_compressed(os.path.join(HERE, f), **arrays)
    for f in ["synth_c1.npz"] + sorted(files):
        print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, "KiB")


if __name__ == "__main__":
    main()
