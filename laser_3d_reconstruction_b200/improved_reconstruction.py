"""ImprovedLaserReconstructor with the reference's API (improved_reconstruction.py): laser pixels +
disparity map -> 3D, per-point work in libl3d.so (csrc/recon.cu).  No CPU fallback."""
from typing import List, Tuple

import numpy as np

from . import _native as N


class ImprovedLaserReconstructor:
    def __init__(self, Q_matrix: np.ndarray, device=0, verbose=True):
        """:17-35: fx = Q[2,3], baseline = 1/Q[3,2], cx = -Q[0,3], cy = -Q[1,3]."""
        self.Q = Q_matrix
        self.fx = Q_matrix[2, 3]
        self.baseline = 1.0 / Q_matrix[3, 2]
        self.cx = -Q_matrix[0, 3]
        self.cy = -Q_matrix[1, 3]
        self.device = device
        if verbose:
            print(f"ImprovedLaserReconstructor 初始化: fx {self.fx:.2f}, 基线 {self.baseline:.4f}m, "
                  f"主点 ({self.cx:.2f}, {self.cy:.2f})")

    def recon_params(self, kind, min_disparity=1.0, window=3):
        """The N.ReconParams of a DISPARITY kind with this camera's fx, baseline, cx, cy: what l3d_reconstruct and the
        frame pipeline (make_pipeline_config(recon=...)) take."""
        p = N.ReconParams()
        p.kind = kind
        p.fx, p.baseline, p.cx, p.cy = float(self.fx), float(self.baseline), float(self.cx), float(self.cy)
        p.min_disparity = float(min_disparity)
        p.window = int(window)
        p.n_water = 1.33
        return p

    def _run(self, kind, laser_points, disparity_map, min_disparity, window=3):
        if len(laser_points) == 0:
            return np.array([])
        disp = np.asarray(disparity_map)
        if disp.ndim != 2:
            raise ValueError("disparity_map must be HxW")
        xy = N.points_to_array(laser_points)
        out = N.default_context(self.device).reconstruct(self.recon_params(kind, min_disparity, window), xy,
                                                         disp.astype(np.float32, copy=False))
        return out.astype(np.float32) if len(out) else np.array([])

    def reconstruct_from_disparity(self, laser_points: List[Tuple[float, float]], disparity_map: np.ndarray,
                                   min_disparity: float = 1.0) -> np.ndarray:
        """:37-86."""
        return self._run(N.RECON_DISPARITY, laser_points, disparity_map, min_disparity)

    def reconstruct_with_interpolation(self, laser_points: List[Tuple[float, float]], disparity_map: np.ndarray,
                                       window_size: int = 3, min_disparity: float = 1.0) -> np.ndarray:
        """:88-152: median of the valid disparities in the window around each laser pixel."""
        if window_size < 1 or window_size > 9 or not (window_size & 1):
            raise ValueError("window_size must be odd and <= 9")
        return self._run(N.RECON_DISPARITY_MEDIAN, laser_points, disparity_map, min_disparity, window_size)

    def create_laser_depth_map(self, laser_points: List[Tuple[float, float]], disparity_map: np.ndarray,
                               image_shape: Tuple[int, int]) -> np.ndarray:
        """:154-186: depth only at the (rounded) laser pixels with `disparity > 1.0`, one scatter kernel
        (l3d_laser_depth_map); bounds follow `image_shape` like the reference's."""
        h, w = image_shape
        disp = np.asarray(disparity_map, np.float32)
        if disp.shape[0] < h or disp.shape[1] < w:
            raise IndexError("disparity_map smaller than image_shape")  # the reference indexes out of bounds here
        if len(laser_points) == 0:
            return np.zeros((h, w), np.float32)
        return N.default_context(self.device).laser_depth_map(laser_points, np.ascontiguousarray(disp[:h, :w]), float(self.fx), float(self.baseline))


def fix_roi_alignment(left_rect, right_rect, roi_left, roi_right):
    """:189-227 -- pure slicing (host)."""
    x1, y1 = max(roi_left[0], roi_right[0]), max(roi_left[1], roi_right[1])
    x2 = min(roi_left[0] + roi_left[2], roi_right[0] + roi_right[2])
    y2 = min(roi_left[1] + roi_left[3], roi_right[1] + roi_right[3])
    if x2 - x1 > 0 and y2 - y1 > 0:
        return left_rect[y1:y2, x1:x2], right_rect[y1:y2, x1:x2]
    return left_rect, right_rect


def visualize_laser_depth(image, laser_points, depth_map, max_depth: float = 5.0):
    """:230-279 -- host-side drawing for the demo windows: every laser point with a positive depth becomes a radius-2 dot in
    the reference's four-segment colour ramp (near = blue-ish in BGR order, far = red-ish) on a copy of the image, and a
    single pixel of a black image of the same size.  -> (vis, depth_colored)"""
    import cv2
    vis = image.copy()
    h, w = image.shape[:2]
    depth_colored = np.zeros((h, w, 3), dtype=np.uint8)
    for x, y in laser_points:
        px, py = int(round(x)), int(round(y))
        if px < 0 or px >= w or py < 0 or py >= h:
            continue
        depth = depth_map[py, px]
        if not depth > 0:
            continue
        t = np.clip(depth / max_depth, 0, 1)
        if t < 0.25:
            color = (255, int(t * 4 * 255), 0)
        elif t < 0.5:
            color = (int((0.5 - t) * 4 * 255), 255, 0)
        elif t < 0.75:
            color = (0, 255, int((t - 0.5) * 4 * 255))
        else:
            color = (0, int((1 - t) * 4 * 255), 255)
        cv2.circle(vis, (px, py), 2, color, -1)
        depth_colored[py, px] = color
    return vis, depth_colored
