"""Reconstructor with the reference's API (core/reconstruction.py); the per-point arithmetic
(ray / laser-plane intersection, Snell refraction, depth back-projection) runs in libl3d.so
(csrc/recon.cu), f64 like the reference.  No CPU fallback.

filter_outliers / transform_points / merge_point_clouds (:184-261) are point-cloud post-processing,
outside the per-frame hot path (SURVEY section 2, row 4): kept as plain numpy with the reference's
semantics so that callers keep working.
"""
from typing import List, NamedTuple, Tuple

import numpy as np

from .. import _native as N


class Reconstructor:
    def __init__(self, camera_intrinsic: np.ndarray, laser_plane: np.ndarray, use_refraction_correction: bool = True,
                 device=0):
        self.K = camera_intrinsic
        self.K_inv = np.linalg.inv(camera_intrinsic)
        self.laser_plane = laser_plane
        self.use_refraction = use_refraction_correction
        self.water_refraction_index = 1.33
        self.device = device

    def _params(self, kind):
        p = N.ReconParams()
        p.kind = kind
        p.K[:] = [float(v) for v in np.asarray(self.K, np.float64).reshape(9)]
        p.plane[:] = [float(v) for v in np.asarray(self.laser_plane, np.float64).reshape(4)]
        p.use_refraction = int(bool(self.use_refraction))
        p.n_water = float(self.water_refraction_index)
        return p

    @staticmethod
    def _points(laser_points):
        return N.points_to_array(laser_points)

    def reconstruct_point(self, u: float, v: float) -> np.ndarray:
        """:30-70 -> [x, y, z], NaN when the ray misses the plane."""
        out = N.default_context(self.device).reconstruct(self._params(N.RECON_PLANE), [(float(u), float(v))])
        return out[0].copy() if len(out) else np.array([np.nan, np.nan, np.nan])

    def reconstruct_laser_line(self, laser_points: List[Tuple[float, float]]) -> np.ndarray:
        """:121-143."""
        if len(laser_points) == 0:
            return np.array([])
        out = N.default_context(self.device).reconstruct(self._params(N.RECON_PLANE), self._points(laser_points))
        return out.copy() if len(out) else np.array([])

    def reconstruct_from_depth(self, laser_points: List[Tuple[float, float]], depth_image: np.ndarray) -> np.ndarray:
        """:145-182 (the depth/1000 unit quirk is preserved)."""
        if len(laser_points) == 0:
            return np.array([])
        depth = np.asarray(depth_image)
        if depth.ndim != 2:
            raise ValueError("depth_image must be HxW")
        out = N.default_context(self.device).reconstruct(self._params(N.RECON_DEPTH), self._points(laser_points),
                                                         depth.astype(np.float32, copy=False))
        return out.copy() if len(out) else np.array([])

    # ---- post-processing helpers, host-side (out of the hot path) ---------------------------
    def filter_outliers(self, points_3d: np.ndarray, threshold: float = 0.01) -> np.ndarray:
        """:184-219: keep points whose neighbours in list order are closer than threshold."""
        n = len(points_3d)
        if n < 3:
            return points_3d
        p = np.asarray(points_3d)
        d = np.linalg.norm(p[1:] - p[:-1], axis=1)
        keep = np.zeros(n, bool)
        keep[1:-1] = (d[:-1] < threshold) & (d[1:] < threshold)
        keep[0] = d[0] < threshold
        keep[-1] = d[-1] < threshold
        return p[keep] if keep.any() else np.array([])

    def transform_points(self, points_3d: np.ndarray, R: np.ndarray, t: np.ndarray) -> np.ndarray:
        """:221-238."""
        if len(points_3d) == 0:
            return points_3d
        return (R @ points_3d.T).T + t

    def merge_point_clouds(self, clouds: List[np.ndarray]) -> np.ndarray:
        """:240-261."""
        valid = [c for c in (clouds or []) if len(c) > 0]
        return np.vstack(valid) if valid else np.array([])


class LaserPlaneFit(NamedTuple):
    """Result of fit_laser_plane."""
    plane: np.ndarray        # (4,) float64 a, b, c, d: unit normal, d >= 0 (Reconstructor's laser_plane)
    inlier_mask: np.ndarray  # (n,) bool: the points within `threshold` of `plane`
    inliers: int
    rms: float               # sqrt(mean squared residual) over the inliers, metres
    spread: float            # sqrt(eig[1] / eig[2]) of the inliers' covariance: ~0 for points along one line
    hypothesis: int          # the winning RANSAC hypothesis and its inlier count
    hypothesis_inliers: int


def fit_laser_plane(points, threshold: float = 0.005, hypotheses: int = 1024, seed: int = 0, device=0) -> LaserPlaneFit:
    """The laser plane a x + b y + c z + d = 0 through 3D laser points (n x 3, metres, in the rectified left camera's
    frame), robust to outliers: RANSAC with `hypotheses` planes through point triples drawn from `seed`, then
    least-squares refits on the points within `threshold` metres (l3d_fit_plane, on the GPU).

    Raises ValueError when the points do not determine a usable plane: when they lie close to one line (the laser line
    recorded at one distance, on one flat surface) or when the plane passes through the camera's optical centre, where
    no laser pixel can be triangulated."""
    r = N.default_context(device).fit_plane(points, threshold, hypotheses, seed)
    eig = r["eig"]
    spread = float(np.sqrt(max(eig[1], 0.0) / eig[2])) if eig[2] > 0 else 0.0
    if not spread >= 0.01:
        raise ValueError("the laser points are nearly collinear (spread %.3g < 0.01): they do not determine a plane. Record "
                         "the laser line on surfaces at several distances from the camera, e.g. a board moved through the "
                         "working range, so that the line sweeps across the laser plane" % spread)
    plane = r["plane"]
    if abs(plane[3]) < 1e-6:
        raise ValueError("the fitted laser plane passes through the camera's optical centre (|d| = %.3g m < 1e-6 m): no laser "
                         "pixel can be triangulated against it. The laser must be mounted off the camera's centre"
                         % abs(plane[3]))
    return LaserPlaneFit(plane, r["inlier_mask"], r["inliers"], r["rms"], spread, r["hypothesis"],
                         r["hypothesis_inliers"])
