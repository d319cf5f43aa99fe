"""ctypes binding of libl3d.so (include/l3d.h).

There is NO CPU fallback: if the shared library is missing it is built with nvcc; if that fails, or
if no CUDA device is visible when a context is requested, an exception is raised.
"""
import ctypes as C
import itertools
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libl3d.so")
_lib = None
_lock = threading.Lock()


class L3DError(RuntimeError):
    pass


class SgbmParams(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        "minDisparity", "numDisparities", "blockSize", "P1", "P2", "disp12MaxDiff",
        "preFilterCap", "uniquenessRatio", "speckleWindowSize", "speckleRange", "mode")]


class BmParams(C.Structure):
    """cv2.StereoBM parameters (include/l3d.h: l3d_bm_params)."""
    _fields_ = [(n, C.c_int) for n in (
        "minDisparity", "numDisparities", "blockSize", "preFilterCap", "textureThreshold", "uniquenessRatio",
        "speckleWindowSize", "speckleRange", "disp12MaxDiff")]


class WlsParams(C.Structure):
    _fields_ = [("lambda_", C.c_double), ("sigma_color", C.c_double), ("min_disp", C.c_int),
                ("num_disp", C.c_int), ("dd_radius", C.c_int), ("lrc_thresh", C.c_int),
                ("solver", C.c_int), ("variant", C.c_int)]


WLS_SOLVER_PARALLEL, WLS_SOLVER_SERIAL = 0, 1
WLS_LAMBDA_PER_PASS, WLS_LRC_OUTSIDE_ZERO, WLS_BOX_FULL_IMAGE, WLS_CONF_CLAMP_1 = 1, 2, 4, 8


class DepthConfig(C.Structure):
    _fields_ = [("left", SgbmParams), ("right", SgbmParams), ("wls", WlsParams),
                ("use_wls", C.c_int), ("use_maps", C.c_int), ("use_Q", C.c_int), ("Q", C.c_double * 16)]


class StegerParams(C.Structure):
    _fields_ = [("variant", C.c_int), ("sigma", C.c_double), ("bright_thr", C.c_int),
                ("resp_thr", C.c_double), ("roi", C.c_int * 4), ("hsv_lo", C.c_int * 3), ("hsv_hi", C.c_int * 3)]


class ReconParams(C.Structure):
    _fields_ = [("kind", C.c_int), ("K", C.c_double * 9), ("plane", C.c_double * 4),
                ("use_refraction", C.c_int), ("n_water", C.c_double), ("fx", C.c_double),
                ("baseline", C.c_double), ("cx", C.c_double), ("cy", C.c_double),
                ("min_disparity", C.c_double), ("window", C.c_int)]


class PipelineConfig(C.Structure):
    _fields_ = [("W", C.c_int), ("H", C.c_int), ("depth", DepthConfig), ("extractor", C.c_int),
                ("steger", StegerParams), ("simple_hsv_lo", C.c_int * 3), ("simple_hsv_hi", C.c_int * 3),
                ("simple_bright_thr", C.c_int), ("simple_min_area", C.c_double), ("recon", ReconParams),
                ("max_points", C.c_int), ("lanes", C.c_int)]


STEGER_FAST, STEGER_IMPROVED, STEGER_OPTIMIZED, STEGER_HYBRID = 0, 1, 2, 3
EXTRACT_SIMPLE = 4
RECON_PLANE, RECON_DEPTH, RECON_DISPARITY, RECON_DISPARITY_MEDIAN = 0, 1, 2, 3

EXPORTS = (
    "l3d_ctx_create l3d_ctx_destroy l3d_last_error l3d_sync l3d_device_count l3d_version l3d_launch_count "
    "l3d_set_rectify_maps l3d_init_undistort_rectify_map l3d_remap_gray l3d_bgr2gray l3d_sgbm_compute l3d_sgbm_compute_pair l3d_sgbm_debug l3d_sgbm_volume_rows "
    "l3d_sgbm_vgroup_time l3d_bm_compute l3d_median3_s16 l3d_filter_speckles l3d_wls_filter l3d_fgs_solve l3d_disp_to_depth l3d_compute_depth "
    "l3d_simple_extract l3d_colour_mask l3d_steger_extract l3d_reconstruct l3d_laser_depth_map l3d_voxel_downsample l3d_statistical_outlier_removal l3d_pipeline_create l3d_pipeline_destroy "
    "l3d_pipeline_set_maps l3d_pipeline_run_dev l3d_pipeline_run_host l3d_pipeline_fetch l3d_pipeline_fetch_points l3d_pipeline_points_needed "
    "l3d_pipeline_pack_points_dev l3d_pipeline_launch_count l3d_pipeline_graph_replays l3d_pipeline_last_ms l3d_pipeline_set_timing l3d_pipeline_kernel_time "
    "l3d_host_alloc l3d_host_free l3d_dev_alloc l3d_dev_free l3d_memcpy_h2d l3d_memcpy_d2h"
).split()


def lib_path():
    return _LIB_PATH


def load():
    """Load (building if necessary) libl3d.so.  Raises if it cannot be produced."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(_LIB_PATH):
            from . import build as _b
            _b.build()
        # one hardware work queue per pipeline stream (read by the driver when the CUDA context is created)
        os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
        lib = C.CDLL(_LIB_PATH)
        for name in EXPORTS:
            if not hasattr(lib, name):
                raise L3DError("libl3d.so does not export %s" % name)
        lib.l3d_last_error.restype = C.c_char_p
        lib.l3d_version.restype = C.c_char_p
        lib.l3d_launch_count.restype = C.c_longlong
        lib.l3d_pipeline_launch_count.restype = C.c_longlong
        lib.l3d_pipeline_graph_replays.restype = C.c_longlong
        lib.l3d_pipeline_graph_replays.argtypes = [C.c_void_p]
        lib.l3d_pipeline_last_ms.restype = C.c_float
        lib.l3d_host_alloc.restype = C.c_void_p
        lib.l3d_host_alloc.argtypes = [C.c_long]
        lib.l3d_host_free.argtypes = [C.c_void_p]
        lib.l3d_dev_alloc.restype = C.c_void_p
        lib.l3d_dev_alloc.argtypes = [C.c_void_p, C.c_long]
        lib.l3d_dev_free.argtypes = [C.c_void_p, C.c_void_p]
        lib.l3d_memcpy_h2d.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_long]
        lib.l3d_memcpy_d2h.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_long]
        lib.l3d_ctx_destroy.argtypes = [C.c_void_p]
        lib.l3d_last_error.argtypes = [C.c_void_p]
        lib.l3d_sync.argtypes = [C.c_void_p]
        lib.l3d_launch_count.argtypes = [C.c_void_p]
        lib.l3d_pipeline_destroy.argtypes = [C.c_void_p]
        lib.l3d_pipeline_launch_count.argtypes = [C.c_void_p]
        lib.l3d_pipeline_last_ms.argtypes = [C.c_void_p]
        _lib = lib
        return lib


def _ptr(a):
    if a is None:
        return None
    return a.ctypes.data_as(C.c_void_p)


def _arr(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


def _rows_u8c3(a):
    """HxWx3 uint8 image whose ROWS may be strided (the views `_split_frame` returns: frame[:, :mid], frame[:, mid:]):
    returned as it is -- the C ABI takes a row stride, so the side-by-side split costs no copy.  Anything else is made
    contiguous."""
    a = np.asarray(a)
    if (a.dtype == np.uint8 and a.ndim == 3 and a.shape[2] == 3 and a.strides[2] == 1 and a.strides[1] == 3
            and a.strides[0] >= 3 * a.shape[1]):
        return a
    return np.ascontiguousarray(a, dtype=np.uint8)


class Context:
    """One GPU context (stream + scratch).  Not thread-safe; create one per thread."""

    def __init__(self, device=0):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.l3d_ctx_create(int(device), C.byref(h))
        if rc != 0:
            msg = self.lib.l3d_last_error(None).decode()
            raise L3DError("l3d_ctx_create(device=%d) failed (%d): %s" % (device, rc, msg))
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.l3d_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc, what):
        if rc != 0:
            raise L3DError("%s failed (%d): %s" % (what, rc, self.lib.l3d_last_error(self.h).decode()))

    @property
    def launches(self):
        return int(self.lib.l3d_launch_count(self.h))

    # ---- stage wrappers (host numpy in / out) ---------------------------------------------
    def init_undistort_rectify_map(self, K, dist, R, P, size):
        """cv2.initUndistortRectifyMap(K, dist, R, P, size, cv2.CV_32FC1) -> (mapx, mapy), computed on the GPU."""
        W, H = int(size[0]), int(size[1])
        K = np.ascontiguousarray(K, np.float64).reshape(3, 3)
        d = np.ascontiguousarray(np.asarray(dist, np.float64).ravel()) if dist is not None else np.zeros(0)
        A = np.asarray(P, np.float64)[:3, :3] if P is not None else K
        Rm = np.asarray(R, np.float64).reshape(3, 3) if R is not None else np.eye(3)
        iR = np.ascontiguousarray(np.linalg.inv(A @ Rm))
        mapx, mapy = np.empty((H, W), np.float32), np.empty((H, W), np.float32)
        self.check(self.lib.l3d_init_undistort_rectify_map(self.h, _ptr(K), _ptr(d) if d.size else None, int(d.size), _ptr(iR),
                                                           W, H, _ptr(mapx), _ptr(mapy)), "l3d_init_undistort_rectify_map")
        return mapx, mapy

    def set_rectify_maps(self, eye, mapx, mapy):
        mapx, mapy = _arr(mapx, np.float32), _arr(mapy, np.float32)
        if mapx.shape != mapy.shape or mapx.ndim != 2:
            raise ValueError("rectification maps must be two HxW float32 arrays")
        H, W = mapx.shape
        self.check(self.lib.l3d_set_rectify_maps(self.h, int(eye), _ptr(mapx), _ptr(mapy), W, H), "l3d_set_rectify_maps")
        return W, H

    def remap_gray(self, eye, src_bgr, out_shape):
        src = _rows_u8c3(src_bgr)
        if src.ndim != 3 or src.shape[2] != 3:
            raise ValueError("remap_gray expects an HxWx3 uint8 image")
        H, W = out_shape
        rect = np.empty((H, W, 3), np.uint8)
        gray = np.empty((H, W), np.uint8)
        self.check(self.lib.l3d_remap_gray(self.h, int(eye), _ptr(src), src.shape[1], src.shape[0],
                                           C.c_long(src.strides[0]), _ptr(rect), _ptr(gray)), "l3d_remap_gray")
        return rect, gray

    def bgr2gray(self, bgr):
        bgr = _arr(bgr, np.uint8)
        out = np.empty(bgr.shape[:2], np.uint8)
        self.check(self.lib.l3d_bgr2gray(self.h, _ptr(bgr), bgr.shape[1], bgr.shape[0], _ptr(out)), "l3d_bgr2gray")
        return out

    def voxel_downsample(self, points, voxel_size):
        """PointCloudProcessor.voxel_downsample without Open3D (utils/point_cloud.py:54-78) on the GPU."""
        f32 = np.asarray(points).dtype == np.float32  # numpy then works in float32 (main.py:208 hands over such a cloud)
        pts = np.ascontiguousarray(points, np.float64).reshape(-1, 3)
        out = np.empty_like(pts)
        m = C.c_int(0)
        self.check(self.lib.l3d_voxel_downsample(self.h, _ptr(pts), int(pts.shape[0]), C.c_double(float(voxel_size)), int(f32),
                                                 _ptr(out), C.byref(m)), "l3d_voxel_downsample")
        res = out[:m.value]
        return res.astype(np.float32) if f32 else res.copy()

    def statistical_outlier_removal(self, points, nb_neighbors, std_ratio):
        """PointCloudProcessor.statistical_outlier_removal without Open3D (utils/point_cloud.py:108-131) on the GPU."""
        f32 = np.asarray(points).dtype == np.float32  # cKDTree promotes to f64 exactly; the kept rows keep their dtype
        pts = np.ascontiguousarray(points, np.float64).reshape(-1, 3)
        out = np.empty_like(pts)
        m = C.c_int(0)
        self.check(self.lib.l3d_statistical_outlier_removal(self.h, _ptr(pts), int(pts.shape[0]), int(nb_neighbors),
                                                            C.c_double(float(std_ratio)), _ptr(out), C.byref(m)),
                   "l3d_statistical_outlier_removal")
        res = out[:m.value]
        return res.astype(np.float32) if f32 else res.copy()

    def bm_compute(self, params, left, right):
        """cv2.StereoBM.compute(left, right) -> int16 disparity x16 (include/l3d.h: l3d_bm_compute)."""
        left, right = _arr(left, np.uint8), _arr(right, np.uint8)
        if left.ndim != 2 or left.shape != right.shape:
            raise ValueError("StereoBM.compute expects two single-channel uint8 images of equal size")
        H, W = left.shape
        disp = np.empty((H, W), np.int16)
        self.check(self.lib.l3d_bm_compute(self.h, C.byref(params), _ptr(left), _ptr(right), W, H, _ptr(disp)), "l3d_bm_compute")
        return disp

    def sgbm_compute(self, params, left, right, want_raw=False, want_volumes=False):
        left, right = _arr(left, np.uint8), _arr(right, np.uint8)
        if left.ndim != 2 or left.shape != right.shape:
            raise ValueError("StereoSGBM.compute expects two single-channel uint8 images of equal size")
        H, W = left.shape
        disp = np.empty((H, W), np.int16)
        raw = np.empty((H, W), np.int16) if want_raw else None
        Cv = Sv = None
        if want_volumes:
            hv = self.lib.l3d_sgbm_volume_rows(C.byref(params), W, H)
            if hv <= 0:
                raise L3DError("unsupported StereoSGBM parameters")
            minD, D = params.minDisparity, params.numDisparities
            width1 = max((W + min(minD, 0)) - max(minD + D, 0), 0)
            Cv = np.zeros((hv, width1, D), np.int16)
            Sv = np.zeros((hv, width1, D), np.int16)
        self.check(self.lib.l3d_sgbm_debug(self.h, C.byref(params), _ptr(left), _ptr(right), W, H, _ptr(disp),
                                           _ptr(raw), _ptr(Cv), _ptr(Sv)), "l3d_sgbm_compute")
        out = [disp]
        if want_raw:
            out.append(raw)
        if want_volumes:
            out += [Cv, Sv]
        return out[0] if len(out) == 1 else tuple(out)

    def sgbm_compute_pair(self, params_left, params_right, left, right, want_volumes=False):
        """stereo_matcher.compute(left, right) and right_matcher.compute(right, left) in one call (shared BT operands
        and, where covered, one pixel-cost pass for both cost volumes).  -> (disp_left, disp_right[, C_left, C_right])"""
        left, right = _arr(left, np.uint8), _arr(right, np.uint8)
        if left.ndim != 2 or left.shape != right.shape:
            raise ValueError("StereoSGBM.compute expects two single-channel uint8 images of equal size")
        H, W = left.shape
        dl, dr = np.empty((H, W), np.int16), np.empty((H, W), np.int16)
        vols = [None, None]
        if want_volumes:
            for i, p in enumerate((params_left, params_right)):
                hv = self.lib.l3d_sgbm_volume_rows(C.byref(p), W, H)
                if hv <= 0:
                    raise L3DError("unsupported StereoSGBM parameters")
                minD, D = p.minDisparity, p.numDisparities
                width1 = (W + min(minD, 0)) - max(minD + D, 0)
                vols[i] = np.zeros((hv, max(width1, 0), D), np.int16)
        self.check(self.lib.l3d_sgbm_compute_pair(self.h, C.byref(params_left), C.byref(params_right), _ptr(left), _ptr(right),
                                                  W, H, _ptr(dl), _ptr(dr), _ptr(vols[0]), _ptr(vols[1])),
                   "l3d_sgbm_compute_pair")
        return (dl, dr, vols[0], vols[1]) if want_volumes else (dl, dr)

    def median3_s16(self, a):
        a = _arr(a, np.int16)
        out = np.empty_like(a)
        self.check(self.lib.l3d_median3_s16(self.h, _ptr(a), a.shape[1], a.shape[0], _ptr(out)), "l3d_median3_s16")
        return out

    def filter_speckles(self, a, new_val, max_size, max_diff):
        a = _arr(a, np.int16).copy()
        self.check(self.lib.l3d_filter_speckles(self.h, _ptr(a), a.shape[1], a.shape[0], int(new_val), int(max_size),
                                                int(max_diff)), "l3d_filter_speckles")
        return a

    def wls_filter(self, params, dl, dr, guide, want_conf=False):
        dl, dr, guide = _arr(dl, np.int16), _arr(dr, np.int16), _arr(guide, np.uint8)
        if dl.shape != dr.shape or dl.shape != guide.shape[:2] or guide.ndim != 2:
            raise ValueError("wls filter expects int16 disparities and a single-channel guide of equal size")
        H, W = dl.shape
        out = np.empty((H, W), np.int16)
        conf = np.empty((H, W), np.float32) if want_conf else None
        self.check(self.lib.l3d_wls_filter(self.h, C.byref(params), _ptr(dl), _ptr(dr), _ptr(guide), W, H, _ptr(out),
                                           _ptr(conf)), "l3d_wls_filter")
        return (out, conf) if want_conf else out

    def fgs_solve(self, num, den, ch, cv, lam=8000.0, iters=3, variant=0, solver=WLS_SOLVER_PARALLEL):
        """The FGS passes of wls_filter alone (include/l3d.h: l3d_fgs_solve) on h x w float32 planes: num / den solved
        with row weights ch and column weights cv.  -> (num, den, parallel_used)"""
        num, den = _arr(num, np.float32).copy(), _arr(den, np.float32).copy()
        ch, cv = _arr(ch, np.float32), _arr(cv, np.float32)
        if num.ndim != 2 or not (num.shape == den.shape == ch.shape == cv.shape):
            raise ValueError("fgs_solve expects four float32 planes of equal 2-D shape")
        H, W = num.shape
        par = C.c_int(-1)
        self.check(self.lib.l3d_fgs_solve(self.h, int(solver), int(variant), C.c_double(lam), int(iters), _ptr(ch), _ptr(cv),
                                          W, H, _ptr(num), _ptr(den), C.byref(par)), "l3d_fgs_solve")
        return num, den, bool(par.value)

    def disp_to_depth(self, disp16, Q=None):
        disp16 = _arr(disp16, np.int16)
        out = np.empty(disp16.shape, np.float32)
        q = _arr(Q, np.float64).reshape(16) if Q is not None else None
        self.check(self.lib.l3d_disp_to_depth(self.h, _ptr(disp16), disp16.shape[1], disp16.shape[0], _ptr(q), _ptr(out)),
                   "l3d_disp_to_depth")
        return out

    def compute_depth(self, cfg, left_bgr, right_bgr, want_disp=False):
        l, r = _rows_u8c3(left_bgr), _rows_u8c3(right_bgr)
        if l.ndim != 3 or l.shape[2] != 3 or l.shape != r.shape:
            raise ValueError("compute_depth expects two HxWx3 uint8 images of equal size")
        if l.strides[0] != r.strides[0]:  # one row stride for both views in the ABI
            l, r = _arr(l, np.uint8), _arr(r, np.uint8)
        H, W = l.shape[:2]
        rect = np.empty((H, W, 3), np.uint8)
        depth = np.empty((H, W), np.float32)
        disp = np.empty((H, W), np.int16) if want_disp else None
        self.check(self.lib.l3d_compute_depth(self.h, C.byref(cfg), _ptr(l), _ptr(r), W, H, C.c_long(l.strides[0]), _ptr(rect),
                                              _ptr(depth), _ptr(disp)), "l3d_compute_depth")
        return (rect, depth, disp) if want_disp else (rect, depth)

    def colour_mask(self, bgr, hsv_lo, hsv_hi, bright_thr=-1):
        """inRange(HSV) & (gray > bright_thr) as a 0/255 mask (core/laser_extractor.py:56-64)"""
        bgr = _arr(bgr, np.uint8)
        if bgr.ndim != 3 or bgr.shape[2] != 3:
            raise ValueError("expects an HxWx3 BGR uint8 image")
        H, W = bgr.shape[:2]
        lo = (C.c_int * 3)(*[int(v) for v in hsv_lo])
        hi = (C.c_int * 3)(*[int(v) for v in hsv_hi])
        mask = np.empty((H, W), np.uint8)
        self.check(self.lib.l3d_colour_mask(self.h, _ptr(bgr), W, H, lo, hi, int(bright_thr), _ptr(mask)), "l3d_colour_mask")
        return mask

    def laser_depth_map(self, xy, disp, fx, baseline):
        """ImprovedLaserReconstructor.create_laser_depth_map (improved_reconstruction.py:154-186)"""
        disp = _arr(disp, np.float32)
        H, W = disp.shape
        xy = _arr(points_to_array(xy), np.float64)
        out = np.empty((H, W), np.float32)
        self.check(self.lib.l3d_laser_depth_map(self.h, _ptr(xy) if len(xy) else None, len(xy), _ptr(disp), W, H,
                                                C.c_double(fx), C.c_double(baseline), _ptr(out)), "l3d_laser_depth_map")
        return out

    def simple_extract(self, bgr, hsv_lo, hsv_hi, bright_thr, min_area, want_masks=False):
        bgr = _arr(bgr, np.uint8)
        if bgr.ndim != 3 or bgr.shape[2] != 3:
            raise ValueError("SimpleLaserExtractor expects an HxWx3 BGR uint8 image")
        H, W = bgr.shape[:2]
        lo = (C.c_int * 3)(*[int(v) for v in hsv_lo])
        hi = (C.c_int * 3)(*[int(v) for v in hsv_hi])
        xy = np.empty((H, 2), np.float64)
        n = C.c_int(0)
        m1 = np.empty((H, W), np.uint8) if want_masks else None
        m2 = np.empty((H, W), np.uint8) if want_masks else None
        self.check(self.lib.l3d_simple_extract(self.h, _ptr(bgr), W, H, lo, hi, int(bright_thr), C.c_double(min_area),
                                               _ptr(m1), _ptr(m2), _ptr(xy), C.byref(n)), "l3d_simple_extract")
        pts = xy[:n.value]
        return (pts, m1, m2) if want_masks else pts

    def steger_extract(self, params, img):
        img = _arr(img, np.uint8)
        channels = 1 if img.ndim == 2 else img.shape[2]
        H, W = img.shape[:2]
        cap = 4 * max(W, H) + 4096
        while True:
            xy = np.empty((cap, 2), np.float32)
            n = C.c_int(0)
            self.check(self.lib.l3d_steger_extract(self.h, C.byref(params), _ptr(img), channels, W, H, _ptr(xy), cap,
                                                   C.byref(n)), "l3d_steger_extract")
            if n.value <= cap:
                return xy[:n.value]
            cap = n.value

    def reconstruct(self, params, xy, img=None):
        xy = _arr(xy, np.float64).reshape(-1, 2)
        n = xy.shape[0]
        out = np.empty((max(n, 1), 3), np.float64)
        n_out = C.c_int(0)
        W = H = 0
        if img is not None:
            img = _arr(img, np.float32)
            H, W = img.shape
        self.check(self.lib.l3d_reconstruct(self.h, C.byref(params), _ptr(xy), n, _ptr(img), W, H, _ptr(out),
                                            C.byref(n_out)), "l3d_reconstruct")
        return out[:n_out.value]


# ---- default contexts: one per (thread, device) ---------------------------------------------
# A Context owns one stream and grow-only scratch buffers and is not thread-safe (include/l3d.h: one l3d_ctx per
# (thread, GPU)), so the reference-API classes -- which share "the" context of their device -- get a separate one in
# every thread that uses them (e.g. a capture thread next to a processing thread).
def points_to_list(pts):
    """(n, 2) array -> list of (x, y) tuples of Python floats, the reference extractors' return type.  Two column
    `tolist()`s zipped: a third faster than building n two-element lists first (0.43 vs 0.63 ms for 4600 points)."""
    a = np.asarray(pts, np.float64).reshape(-1, 2)
    return list(zip(a[:, 0].tolist(), a[:, 1].tolist()))


def points_to_list_f32(pts):
    """(n, 2) float32 array -> list of (np.float32, np.float32) tuples, FastStegerExtractor's return type in the reference
    (core/laser_extractor.py:256 appends the float32 scalars as they are); zip of the two columns, ~9x faster than
    unpacking row by row."""
    a = np.asarray(pts, np.float32).reshape(-1, 2)
    return list(zip(a[:, 0], a[:, 1]))


def points_to_array(points):
    """list of (u, v) pairs (or anything array-like) -> (n, 2) float64.  A list of pairs is flattened by
    `np.fromiter` over one chained iterator (about 2.5x faster than np.asarray on 4600 tuples)."""
    if isinstance(points, (list, tuple)) and len(points) and isinstance(points[0], (tuple, list)):
        try:
            if set(map(len, points)) == {2}:   # every entry a pair: nothing can be mis-grouped by the flat iterator
                return np.fromiter(itertools.chain.from_iterable(points), np.float64, 2 * len(points)).reshape(-1, 2)
        except (TypeError, ValueError):
            pass  # entries without a length or non-numeric: let numpy's own conversion raise or cope
    return np.asarray(points, np.float64).reshape(-1, 2)


_default = threading.local()


def default_context(device=0):
    """The calling thread's Context of `device`, used by the reference-API classes.  Raises L3DError
    when the CUDA library or a GPU is missing: there is no CPU fallback."""
    table = getattr(_default, "ctx", None)
    if table is None:
        table = _default.ctx = {}
    ctx = table.get(device)
    if ctx is None or ctx.h is None:
        ctx = table[device] = Context(device)
    return ctx
