"""Batched, device-resident frame pipeline: LaserReconstructionSystem.process_frame
(reference main.py:164-189) for many independent frames at once, and its frame-wise sharding over
the GPUs of one box (no collective on the hot path; NCCL only gathers the point clouds).

    rectify -> gray -> SGBM left/right -> WLS -> depth -> laser centre line -> 3D points
"""
import ctypes as C
import math
import weakref

import numpy as np

from . import _native as N


def sgbm_params(num_disparities, block_size, mode, min_disparity=0, disp12=1, uniq=10, speckle=(100, 32),
                pre_filter_cap=63):
    """cv2.StereoSGBM_create arguments as the reference builds them
    (camera/single_usb_stereo_camera.py:252-274): P1 = 8*3*bs^2, P2 = 32*3*bs^2."""
    return N.SgbmParams(min_disparity, num_disparities, block_size, 8 * 3 * block_size ** 2,
                        32 * 3 * block_size ** 2, disp12, pre_filter_cap, uniq, speckle[0], speckle[1], mode)


def wls_mutate(p):
    """cv2.ximgproc.createDisparityWLSFilter(left_matcher) mutates the matcher it is given."""
    q = N.SgbmParams.from_buffer_copy(p)
    q.disp12MaxDiff = 1000000
    q.speckleWindowSize = 0
    q.uniquenessRatio = 0
    return q


def right_matcher_params(p):
    """cv2.ximgproc.createRightMatcher(left_matcher) for a StereoSGBM."""
    return N.SgbmParams(-(p.minDisparity + p.numDisparities) + 1, p.numDisparities, p.blockSize, p.P1, p.P2,
                        1000000, p.preFilterCap, 0, 0, 0, p.mode)


def depth_config(num_disparities, block_size, mode, Q, use_wls=True, use_maps=True, lam=8000.0, sigma_color=1.5,
                 mutated_left=False):
    """use_wls=False runs the left matcher alone, with its parameters as constructed; mutated_left=True runs it
    as createDisparityWLSFilter leaves it instead (the Improved/Hybrid order of test_improved_laser.py:112-207).
    With use_wls=True the left matcher is always the mutated one."""
    cfg = N.DepthConfig()
    left = sgbm_params(num_disparities, block_size, mode)
    if use_wls:
        cfg.right = right_matcher_params(left)  # created before the mutation, but identical either way
    if use_wls or mutated_left:
        left = wls_mutate(left)
    cfg.left = left
    cfg.wls = N.WlsParams(lam, sigma_color, left.minDisparity, left.numDisparities, int(math.ceil(0.5 * block_size)), 24)
    cfg.use_wls = int(use_wls)
    cfg.use_maps = int(use_maps)
    cfg.use_Q = int(Q is not None)
    if Q is not None:
        cfg.Q[:] = [float(v) for v in np.asarray(Q, np.float64).reshape(16)]
    return cfg


def make_pipeline_config(W, H, num_disparities, block_size, mode, Q, K, extractor=N.STEGER_IMPROVED, lanes=2,
                         max_points=20000, use_wls=True, use_maps=True, sigma=3.0, bright_thr=200, resp_thr=0.5,
                         hsv_lo=(50, 100, 180), hsv_hi=(70, 255, 255), min_area=50.0, recon=None, mutated_left=False):
    """recon: the per-frame reconstruction as an N.ReconParams.  None (default) is reconstruct_from_depth with
    camera matrix K (main.py:176).  The DISPARITY kinds come from ImprovedLaserReconstructor(Q).recon_params and
    read the frame's int16 disparity (disp16) as disp16 / 16.0."""
    cfg = N.PipelineConfig()
    cfg.W, cfg.H = W, H
    cfg.depth = depth_config(num_disparities, block_size, mode, Q, use_wls, use_maps, mutated_left=mutated_left)
    cfg.extractor = extractor
    cfg.steger = N.StegerParams(min(extractor, 3), sigma, bright_thr, resp_thr, (C.c_int * 4)(0, 0, 0, 0),
                                (C.c_int * 3)(*hsv_lo), (C.c_int * 3)(*hsv_hi))
    cfg.simple_hsv_lo[:] = list(hsv_lo)
    cfg.simple_hsv_hi[:] = list(hsv_hi)
    cfg.simple_bright_thr = bright_thr
    cfg.simple_min_area = min_area
    if recon is None:
        recon = N.ReconParams()
        recon.kind = N.RECON_DEPTH  # main.py:176 calls reconstruct_from_depth
        recon.K[:] = [float(v) for v in np.asarray(K, np.float64).reshape(9)]
        recon.n_water = 1.33
    cfg.recon = recon
    cfg.max_points = max_points
    cfg.lanes = lanes
    return cfg


class FramePipeline:
    """Owns a Context and an l3d_pipeline; frames in, per-frame depth + point clouds out."""

    def __init__(self, cfg, maps=None, device=0, ctx=None):
        self.ctx = ctx or N.Context(device)
        self.cfg = cfg
        self.lib = self.ctx.lib
        self.h = C.c_void_p()
        self.ctx.check(self.lib.l3d_pipeline_create(self.ctx.h, C.byref(cfg), C.byref(self.h)), "l3d_pipeline_create")
        if maps is not None:
            mlx, mly, mrx, mry = [np.ascontiguousarray(m, np.float32) for m in maps]
            self.ctx.check(self.lib.l3d_pipeline_set_maps(self.h, 0, N._ptr(mlx), N._ptr(mly)), "l3d_pipeline_set_maps")
            self.ctx.check(self.lib.l3d_pipeline_set_maps(self.h, 1, N._ptr(mrx), N._ptr(mry)), "l3d_pipeline_set_maps")
        self._dev = []

    def close(self):
        if self.h:
            for p in self._dev:
                self.lib.l3d_dev_free(self.ctx.h, p)
            self._dev = []
            self.lib.l3d_pipeline_destroy(self.h)
            self.h = None

    def upload(self, frames_u8):
        """Stage a (nframes, H, W, 3) uint8 batch in HBM; returns the device pointer."""
        a = np.ascontiguousarray(frames_u8, np.uint8)
        p = self.lib.l3d_dev_alloc(self.ctx.h, a.nbytes)
        if not p:
            raise N.L3DError("device allocation of %d bytes failed" % a.nbytes)
        self.ctx.check(self.lib.l3d_memcpy_h2d(self.ctx.h, p, a.ctypes.data, a.nbytes), "l3d_memcpy_h2d")
        self._dev.append(p)
        return p

    def run_dev(self, left_dev, right_dev, nframes):
        counts = (C.c_int * nframes)()
        self.ctx.check(self.lib.l3d_pipeline_run_dev(self.h, C.c_void_p(left_dev), C.c_void_p(right_dev), nframes, counts),
                       "l3d_pipeline_run_dev")
        return np.frombuffer(counts, np.int32).copy()

    def run_host(self, left, right, depth_out=None, xyz_out=None):
        """left/right: (n,H,W,3) uint8 host arrays (pinned for full overlap); depth_out (n,H,W) float32 and
        xyz_out (n,max_points,3) float64 are optional C-contiguous result buffers."""
        n = left.shape[0]
        want = (n, self.cfg.H, self.cfg.W, 3)
        for name, a in (("left", left), ("right", right)):
            if a.dtype != np.uint8 or a.shape != want or not a.flags.c_contiguous:
                raise N.L3DError("run_host: %s must be a C-contiguous uint8 array of shape %s" % (name, want))
        self._check_outputs("run_host", n, depth_out, xyz_out)
        counts = (C.c_int * n)()
        self.ctx.check(self.lib.l3d_pipeline_run_host(self.h, C.c_void_p(left.ctypes.data), C.c_void_p(right.ctypes.data), n,
                                                      C.c_void_p(depth_out.ctypes.data) if depth_out is not None else None,
                                                      C.c_void_p(xyz_out.ctypes.data) if xyz_out is not None else None,
                                                      counts), "l3d_pipeline_run_host")
        return np.frombuffer(counts, np.int32).copy()

    def capture_shape(self, n, split):
        """Shape of n stereo captures as cap.read() delivers them: (n, H, 2W, 3) side by side (split 0, the camera's
        'horizontal' split_mode) or (n, 2H, W, 3) one above the other (split 1)."""
        if split not in (0, 1):
            raise N.L3DError("split must be 0 (side by side) or 1 (top / bottom), not %r" % (split,))
        W, H = self.cfg.W, self.cfg.H
        return (n, H, 2 * W, 3) if split == 0 else (n, 2 * H, W, 3)

    def run_captures_host(self, frames, split, depth_out=None, xyz_out=None):
        """run_host on stereo captures: frames = (n, H, 2W, 3) (split 0) or (n, 2H, W, 3) (split 1) C-contiguous uint8
        host array (pinned for full overlap), each capture uploaded with one copy and split on the device;
        depth_out / xyz_out as for run_host."""
        frames = np.asarray(frames)
        n = frames.shape[0] if frames.ndim == 4 else 0
        want = self.capture_shape(n, split)
        if frames.dtype != np.uint8 or frames.shape != want or n == 0 or not frames.flags.c_contiguous:
            raise N.L3DError("run_captures_host: frames must be a C-contiguous uint8 array of shape %s" % (want,))
        self._check_outputs("run_captures_host", n, depth_out, xyz_out)
        counts = (C.c_int * n)()
        self.ctx.check(self.lib.l3d_pipeline_run_captures_host(
            self.h, C.c_void_p(frames.ctypes.data), n, int(split),
            C.c_void_p(depth_out.ctypes.data) if depth_out is not None else None,
            C.c_void_p(xyz_out.ctypes.data) if xyz_out is not None else None, counts), "l3d_pipeline_run_captures_host")
        return np.frombuffer(counts, np.int32).copy()

    def run_captures_dev(self, frames_dev, nframes, split):
        """run_dev on nframes stereo captures already in HBM (device pointer to capture_shape(nframes, split) uint8)."""
        self.capture_shape(nframes, split)
        counts = (C.c_int * max(int(nframes), 1))()
        self.ctx.check(self.lib.l3d_pipeline_run_captures_dev(self.h, C.c_void_p(frames_dev), int(nframes), int(split), counts),
                       "l3d_pipeline_run_captures_dev")
        return np.frombuffer(counts, np.int32)[:nframes].copy()

    def _check_outputs(self, what, n, depth_out, xyz_out):
        if depth_out is not None and (depth_out.dtype != np.float32 or not depth_out.flags.c_contiguous
                                      or depth_out.size < n * self.cfg.H * self.cfg.W):
            raise N.L3DError("%s: depth_out must be C-contiguous float32 with room for %d frames" % (what, n))
        if xyz_out is not None and (xyz_out.dtype != np.float64 or not xyz_out.flags.c_contiguous
                                    or xyz_out.size < n * self.cfg.max_points * 3):
            raise N.L3DError("%s: xyz_out must be C-contiguous float64 with room for %d x max_points x 3" % (what, n))

    @property
    def last_ms(self):
        return float(self.lib.l3d_pipeline_last_ms(self.h))

    @property
    def launches(self):
        return int(self.lib.l3d_pipeline_launch_count(self.h))

    @property
    def graph_replays(self):
        """steps replayed as a captured CUDA graph so far (launch-bound repeated steps, see include/l3d.h)"""
        return int(self.lib.l3d_pipeline_graph_replays(self.h))

    def set_timing(self, on):
        self.lib.l3d_pipeline_set_timing(self.h, int(on))

    def kernel_time(self, name):
        t, k = C.c_float(), C.c_int()
        self.ctx.check(self.lib.l3d_pipeline_kernel_time(self.h, name.encode(), C.byref(t), C.byref(k)), "l3d_pipeline_kernel_time")
        return t.value, k.value

    @property
    def points_needed(self):
        """largest 2D point count a frame of the last run produced; > cfg.max_points means truncated point lists"""
        return int(self.lib.l3d_pipeline_points_needed(self.h))

    def fetch(self, frame):
        """Everything frame slot `frame` of the last run produced.  points_2d: float64 for the Simple extractor (its
        exact centroids), float32 for the Steger variants -- the dtypes the reference's extractors return.  points_3d:
        float32 for the DISPARITY kinds (what ImprovedLaserReconstructor returns), float64 otherwise."""
        rect, depth, disp = self.fetch_images(frame, want_disp=True)
        xy, xyz = self.fetch_points(frame, want_2d=True)
        if self.cfg.extractor != N.EXTRACT_SIMPLE:
            xy = xy.astype(np.float32)
        if self.cfg.recon.kind in (N.RECON_DISPARITY, N.RECON_DISPARITY_MEDIAN):
            xyz = xyz.astype(np.float32)
        return dict(left_rect=rect, depth=depth, disp16=disp, points_2d=xy, points_3d=xyz)

    def fetch_images(self, frame, want_disp=False):
        """(left_rect (H,W,3) uint8, depth (H,W) float32) of frame slot `frame` of the last run, in new arrays, and its
        int16 x16 disparity (disp16) as a third element with want_disp."""
        W, H = self.cfg.W, self.cfg.H
        rect = np.empty((H, W, 3), np.uint8)
        depth = np.empty((H, W), np.float32)
        disp = np.empty((H, W), np.int16) if want_disp else None
        self.ctx.check(self.lib.l3d_pipeline_fetch(self.h, int(frame), N._ptr(rect), N._ptr(depth), N._ptr(disp), None,
                                                   None, None, None), "l3d_pipeline_fetch")
        return (rect, depth, disp) if want_disp else (rect, depth)

    def fetch_points(self, frame, want_2d=False):
        """The 3D points (and optionally the 2D centres) of frame slot `frame` of the last run (device -> host);
        buffers are sized from the frame's own counts, clamped to the pipeline's max_points."""
        nxy, nxyz = C.c_int(), C.c_int()
        self.ctx.check(self.lib.l3d_pipeline_fetch_points(self.h, int(frame), None, 0, None, 0, C.byref(nxy), C.byref(nxyz)),
                       "l3d_pipeline_fetch_points")
        cap = self.cfg.max_points
        m2 = min(nxy.value, cap) if want_2d else 0
        m3 = min(nxyz.value, cap)
        xy = np.empty((m2, 2), np.float64)
        xyz = np.empty((m3, 3), np.float64)
        self.ctx.check(self.lib.l3d_pipeline_fetch_points(self.h, int(frame), N._ptr(xy) if m2 else None, m2,
                                                          N._ptr(xyz) if m3 else None, m3, C.byref(nxy), C.byref(nxyz)),
                       "l3d_pipeline_fetch_points")
        return (xy, xyz) if want_2d else xyz

    def pack_points_dev(self, frame_ids, table_ptr):
        """Pack the last run's point clouds into the caller's device table (rows frame_id,x,y,z; f64).
        table_ptr: device pointer with room for sum(counts)*4 doubles.  Returns the number of rows."""
        n = len(frame_ids)
        ids = (C.c_int * n)(*[int(f) for f in frame_ids])
        total = C.c_longlong(0)
        self.ctx.check(self.lib.l3d_pipeline_pack_points_dev(self.h, n, ids, C.c_void_p(table_ptr), C.byref(total)),
                       "l3d_pipeline_pack_points_dev")
        return int(total.value)


def pinned_empty(shape, dtype):
    """numpy array backed by page-locked host memory (l3d_host_alloc)."""
    lib = N.load()
    dtype = np.dtype(dtype)
    nbytes = int(np.prod(shape)) * dtype.itemsize
    p = lib.l3d_host_alloc(max(nbytes, 1))
    if not p:
        raise N.L3DError("pinned allocation of %d bytes failed" % nbytes)
    buf = (C.c_char * nbytes).from_address(p)
    # every view of the array keeps `buf` alive; the block is unpinned with the last one (not at interpreter exit:
    # the CUDA runtime may be gone by then and the process is ending anyway)
    weakref.finalize(buf, lib.l3d_host_free, p).atexit = False
    return np.frombuffer(buf, dtype=dtype).reshape(shape)


from .sharding import shard_frames  # noqa: E402,F401  (frame-wise sharding, SURVEY 8e)
