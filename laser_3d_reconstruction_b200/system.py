"""LaserReconstructionSystem -- the immediate caller of the hot path (reference main.py:40-189, SURVEY 8f N1).

`initialize` / `process_frame` keep the reference's names, flow, prints-and-False error behaviour and
the accumulation rule (rows with a NaN are dropped, main.py:181-184).  `process_frames` is the
batched, device-resident form of the same loop: many already captured stereo pairs go through
`l3d_pipeline_*` (rectify -> SGBM x2 -> WLS -> depth -> extractor -> reconstruct_from_depth without a
host round trip between the stages) and produce exactly what calling `process_frame` once per pair
produces.  `save_point_cloud` (main.py:190-232) runs the point-cloud sink (voxel down-sampling, outlier removal,
PLY) through `utils.PointCloudProcessor`, the GPU form of the reference's Open3D-free code (SURVEY 8f N2).
"""
import itertools

import numpy as np

from . import _native as N
from . import pipeline as _pl
from .camera.single_usb_stereo_camera import SingleUSBStereoCameraManager
from .config import Config
from .core.laser_extractor import FastStegerExtractor, SimpleLaserExtractor
from .core.reconstruction import Reconstructor
from .utils.point_cloud import PointCloudProcessor

# Frames per pipeline call of process_frames: about 1 GB of device results at 1280x720.  Measured on one B200 (1 000 W),
# run_captures_host at 1280x720 in pieces of 28 / 56 / 112 / 224 frames gave 797 / 756 / 758 / 757 frames/s over 448
# frames and 741 / 656 / 807 / 796 over 112 -- no size is faster beyond the noise, and 112 is bench.py's config-3 step.
CHUNK_FRAMES = 112


def _chunks(frames, k):
    """Consecutive pieces of at most k frames: slices of an array, stacked lists of the items of any other iterable."""
    if isinstance(frames, np.ndarray):
        for c0 in range(0, frames.shape[0], k):
            yield frames[c0:c0 + k]
        return
    it = iter(frames)
    while True:
        part = list(itertools.islice(it, k))
        if not part:
            return
        yield np.stack(part)


class LaserReconstructionSystem:
    """reference main.py:40-56 (attributes), :58-162 (initialize), :164-189 (process_frame)."""

    def __init__(self, config=None, verbose=True):
        self.config = config or Config()
        self.camera = None
        self.laser_extractor = None
        self.reconstructor = None
        self.point_cloud_processor = None  # utils.PointCloudProcessor (GPU form of the Open3D-free reference code)
        self.point_cloud = []
        self.frame_count = 0
        self.start_time = None
        self.show_depth = True
        self.verbose = verbose
        self._pipe = None
        self._pipe_key = None
        self._pipe_cap = None

    def _say(self, *a):
        if self.verbose:
            print(*a)

    # ---- reference :58-162 ------------------------------------------------------------------
    def initialize(self, camera_id=None, width=None, height=None, camera=None):
        """`camera`: an already initialised SingleUSBStereoCameraManager (offline / batch use); otherwise the
        capture device is opened like the reference does (returns False without one)."""
        cfg = self.config
        camera_id = camera_id if camera_id is not None else cfg.SINGLE_USB_CAMERA_ID
        width = width or cfg.CAMERA_WIDTH
        height = height or cfg.CAMERA_HEIGHT
        try:
            if camera is not None:
                self.camera = camera
            else:
                self.camera = SingleUSBStereoCameraManager(camera_id=camera_id, width=width, height=height,
                                                           fps=cfg.CAMERA_FPS, split_mode=cfg.SPLIT_MODE,
                                                           calibration_file=cfg.STEREO_CALIBRATION_FILE,
                                                           verbose=self.verbose)
                if not self.camera.initialize():
                    print("❌ 相机初始化失败")
                    return False
        except Exception as e:  # the reference reports and returns False
            print(f"❌ 相机初始化错误: {e}")
            return False
        try:
            if cfg.LASER_EXTRACTOR_TYPE == 'simple':
                self.laser_extractor = SimpleLaserExtractor(hsv_lower=cfg.SIMPLE_LASER_HSV_LOWER,
                                                            hsv_upper=cfg.SIMPLE_LASER_HSV_UPPER,
                                                            brightness_threshold=cfg.SIMPLE_LASER_BRIGHTNESS_THRESHOLD,
                                                            min_area=cfg.SIMPLE_LASER_MIN_AREA)
            else:
                self.laser_extractor = FastStegerExtractor(sigma=cfg.STEGER_SIGMA,
                                                           brightness_threshold=cfg.STEGER_BRIGHTNESS_THRESHOLD,
                                                           use_lut=cfg.STEGER_USE_LUT)
        except Exception as e:
            print(f"❌ 激光提取器初始化错误: {e}")
            return False
        try:
            intr = self.camera.get_camera_intrinsics()
            if intr is None:
                print("❌ 无法获取相机内参")
                return False
            K = np.array([[intr['fx'], 0, intr['cx']], [0, intr['fy'], intr['cy']], [0, 0, 1]], dtype=np.float64)
            self.reconstructor = Reconstructor(camera_intrinsic=K, laser_plane=cfg.LASER_PLANE_COEFFICIENTS,
                                               use_refraction_correction=cfg.USE_REFRACTION_CORRECTION)
        except Exception as e:
            print(f"❌ 重建器初始化错误: {e}")
            return False
        try:
            self.point_cloud_processor = PointCloudProcessor(device=getattr(self.camera, "device", 0), verbose=False)
        except Exception as e:
            print(f"❌ 点云处理器初始化错误: {e}")
            return False
        self._say("✅ 系统初始化完成!")
        return True

    # ---- reference :164-189 -----------------------------------------------------------------
    def process_frame(self):
        color_image, depth_image = self.camera.get_frames()
        if color_image is None:
            return None, None, None
        laser_points = self.laser_extractor.extract_centerline(color_image)
        self._accumulate(laser_points, depth_image)
        self.frame_count += 1
        return color_image, depth_image, laser_points

    def _accumulate(self, laser_points, depth_image):
        if len(laser_points) > 0 and depth_image is not None:
            points_3d = self.reconstructor.reconstruct_from_depth(laser_points, depth_image)
            if len(points_3d) > 0:
                valid_mask = ~np.isnan(points_3d).any(axis=1)
                points_3d = points_3d[valid_mask]
                self.point_cloud.extend(points_3d.tolist())

    # ---- batched, device-resident form ---------------------------------------------------------
    def _pipeline(self, lanes, cap=None):
        cam = self.camera
        W, H = cam.single_width, cam.single_height
        dcfg = cam._depth_config()
        simple = isinstance(self.laser_extractor, SimpleLaserExtractor)
        ex = self.laser_extractor
        cap = max(H, 20000, int(cap or 0))
        key = (W, H, lanes, simple, bytes(dcfg), cap)
        if self._pipe is not None and self._pipe_key == key:
            return self._pipe
        if self._pipe is not None:
            self._pipe.close()
        if simple:
            pc = _pl.make_pipeline_config(W, H, dcfg.left.numDisparities, dcfg.left.blockSize, dcfg.left.mode, None,
                                          self.reconstructor.K, extractor=N.EXTRACT_SIMPLE, lanes=lanes, max_points=cap,
                                          bright_thr=int(ex.brightness_threshold), hsv_lo=tuple(int(v) for v in ex.hsv_lower),
                                          hsv_hi=tuple(int(v) for v in ex.hsv_upper), min_area=float(ex.min_area))
        else:
            pc = _pl.make_pipeline_config(W, H, dcfg.left.numDisparities, dcfg.left.blockSize, dcfg.left.mode, None,
                                          self.reconstructor.K, extractor=N.STEGER_FAST, lanes=lanes, max_points=cap,
                                          sigma=float(ex.sigma), bright_thr=int(ex.brightness_threshold))
        pc.depth = dcfg  # exactly the camera's matcher / WLS / Q configuration
        maps = None
        if dcfg.use_maps:
            maps = (cam.map_left_x, cam.map_left_y, cam.map_right_x, cam.map_right_y)
        self._pipe = _pl.FramePipeline(pc, maps=maps, device=cam.device)
        self._pipe_key = key
        return self._pipe

    def process_frames(self, frames=None, lefts=None, rights=None, lanes=8, want_images=True):
        """Batched `process_frame`: `frames` = stereo captures as `cap.read()` delivers them -- an (n, H, 2W, 3) uint8
        array, or (n, 2H, W, 3) when the camera's split_mode is not 'horizontal' (see `_split_frame`), or a list or other
        iterable of single captures -- or `lefts` / `rights` = already split views (n, H, W, 3).  Returns a list of
        (color_image, depth_image, laser_points) per frame (images omitted when `want_images` is False) and accumulates
        the valid 3D points in `self.point_cloud` in frame order, exactly as n calls of `process_frame` would.

        A C-contiguous uint8 capture array goes to the pipeline as it is: each capture is uploaded with one copy and
        split on the device.  Frames run in chunks of CHUNK_FRAMES, so device memory (about 9 MB per frame at
        1280x720) and the host copy a list is stacked into stay bounded whatever the recording's length."""
        out = []
        if frames is not None:
            split = 0 if self.camera.split_mode == 'horizontal' else 1
            for chunk in _chunks(frames, CHUNK_FRAMES):
                chunk = np.ascontiguousarray(chunk, np.uint8)  # no copy for a slice of a C-contiguous uint8 array
                self._process_chunk(lanes, want_images, out, lambda fp: fp.run_captures_host(chunk, split))
            return out
        lefts = np.ascontiguousarray(lefts, np.uint8)
        rights = np.ascontiguousarray(rights, np.uint8)
        for c0 in range(0, lefts.shape[0], CHUNK_FRAMES):
            l, r = lefts[c0:c0 + CHUNK_FRAMES], rights[c0:c0 + CHUNK_FRAMES]
            self._process_chunk(lanes, want_images, out, lambda fp: fp.run_host(l, r))
        return out

    def _process_chunk(self, lanes, want_images, out, run):
        """One pipeline call (`run(fp)`) over a chunk of frames; its frames' results are appended to `out` and their
        points to `self.point_cloud` only once the chunk has run with room for all of its points."""
        fp = self._pipeline(lanes, self._pipe_cap)
        n = len(run(fp))
        if fp.points_needed > fp.cfg.max_points:
            # a frame found more laser points than the pipeline's point lists hold (FastSteger emits one per bright
            # pixel: a saturated patch can exceed any fixed bound): nothing may be dropped silently -- the single-frame
            # calls grow their buffers too -- so the pipeline is rebuilt with room for them and the chunk runs again
            self._pipe_cap = min(fp.cfg.W * fp.cfg.H, 2 * fp.points_needed)
            fp = self._pipeline(lanes, self._pipe_cap)
            run(fp)
            if fp.points_needed > fp.cfg.max_points:
                raise N.L3DError("process_frames: %d laser points in one frame exceed the point list capacity %d"
                                 % (fp.points_needed, fp.cfg.max_points))
        # np.float64 pairs (Simple) / np.float32 pairs (Steger), as the reference's extractors give them
        to_list = N.points_to_list_f64 if fp.cfg.extractor == N.EXTRACT_SIMPLE else N.points_to_list_f32
        for i in range(n):
            xy, p3 = fp.fetch_points(i, want_2d=True)
            pts2 = to_list(xy)
            if len(p3) > 0:
                p3 = p3[~np.isnan(p3).any(axis=1)]
                self.point_cloud.extend(p3.tolist())
            self.frame_count += 1
            out.append(fp.fetch_images(i) + (pts2,) if want_images else (None, None, pts2))

    # ---- reference :190-232 ---------------------------------------------------------------------
    def save_point_cloud(self, filename=None):
        import time
        from pathlib import Path
        cfg = self.config
        if len(self.point_cloud) < cfg.MIN_POINT_CLOUD_SIZE:
            print(f"⚠️  点云太少 ({len(self.point_cloud)} < {cfg.MIN_POINT_CLOUD_SIZE})，跳过保存")
            return False
        output_dir = Path(cfg.OUTPUT_DIR)
        output_dir.mkdir(exist_ok=True)
        if filename is None:
            filename = f"point_cloud_{time.strftime('%Y%m%d_%H%M%S')}.{cfg.SAVE_FORMAT}"
        filepath = output_dir / filename
        points = np.array(self.point_cloud, dtype=np.float32)
        points = self.point_cloud_processor.voxel_downsample(points, voxel_size=cfg.VOXEL_SIZE)
        points = self.point_cloud_processor.statistical_outlier_removal(points, nb_neighbors=cfg.OUTLIER_REMOVAL_NEIGHBORS,
                                                                        std_ratio=cfg.OUTLIER_REMOVAL_STD_RATIO)
        if cfg.SAVE_FORMAT == 'ply':
            self.point_cloud_processor.save_ply(points, str(filepath))
        else:
            self.point_cloud_processor.save_pcd(points, str(filepath))
        self._say(f"✓ 点云已保存: {filepath}")
        return True

    def run_realtime(self, duration=None, max_frames=None):
        """main.py:235-343 without the windows: the capture -> process_frame loop until `duration` seconds have passed,
        `max_frames` frames have been processed (an addition: a server has no key to press) or Ctrl-C; the accumulated
        cloud is auto-saved every AUTO_SAVE_INTERVAL seconds, and saved once more at the end, as the reference does.
        The reference's OpenCV windows and key handling are a GUI and stay out (DESIGN.md section 7).  -> frames processed"""
        import time
        cfg = self.config
        self.start_time = time.time()
        last_save = time.time()
        try:
            while True:
                if duration and (time.time() - self.start_time) > duration:
                    self._say(f"\n达到设定时长 {duration} 秒")
                    break
                if max_frames is not None and self.frame_count >= max_frames:
                    break
                color_image, depth_image, laser_points = self.process_frame()
                if color_image is None:
                    continue
                if time.time() - last_save > cfg.AUTO_SAVE_INTERVAL and len(self.point_cloud) >= cfg.MIN_POINT_CLOUD_SIZE:
                    self._say("\n自动保存点云...")
                    self.save_point_cloud()
                    last_save = time.time()
        except KeyboardInterrupt:
            self._say("\n检测到键盘中断")
        finally:
            self.stop()
            if len(self.point_cloud) >= cfg.MIN_POINT_CLOUD_SIZE:
                self._say("\n保存最终点云...")
                self.save_point_cloud("final_" + time.strftime("%Y%m%d_%H%M%S") + f".{cfg.SAVE_FORMAT}")
            elapsed = max(time.time() - self.start_time, 1e-9)
            self._say(f"\n重建完成:\n  总帧数: {self.frame_count}\n  总时长: {elapsed:.1f} 秒\n"
                      f"  平均FPS: {self.frame_count / elapsed:.1f}\n  点云大小: {len(self.point_cloud)} 点")
        return self.frame_count

    def stop(self):
        if self._pipe is not None:
            self._pipe.close()
            self._pipe = None
        if self.camera is not None:
            self.camera.stop()
