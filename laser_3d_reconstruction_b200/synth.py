"""Deterministic synthetic input generator (SURVEY.md section 8d).

Rendered, textured, rectified stereo pairs from a known disparity map, with a Gaussian-profile
green laser stripe, plus a smooth lens-like warp so the rectification remap does real work.
Used by tests/, bench.py and __graft_entry__.smoke(); nothing here touches the GPU.
"""
import cv2
import numpy as np


def disparity_field(W, H, D):
    xs = np.arange(W, dtype=np.float64)[None, :]
    ys = np.arange(H, dtype=np.float64)[:, None]
    return 0.35 * D + 0.20 * D * np.sin(6 * xs / W) * np.cos(4 * ys / H)


def stereo_pair(W, H, D, seed=0, laser=True):
    """Returns (left_bgr, right_bgr) uint8 HxWx3: textured scene + green laser stripe."""
    rng = np.random.default_rng(seed)
    pad = D + 16
    tex = rng.integers(0, 256, (H, W + 2 * pad, 3)).astype(np.float32)
    tex = cv2.GaussianBlur(tex, (0, 0), 1.5)
    tex = np.clip((tex - 128.0) * 2.2 + 110.0, 0, 200)  # background never passes gray > 200
    d = disparity_field(W, H, D)
    di = np.rint(d).astype(np.int64)
    xs = np.arange(W)[None, :]
    ys = np.arange(H)[:, None]
    left = tex[ys, xs + pad].copy()
    right = tex[ys, xs + pad + di].copy()
    if laser:
        cx = 0.55 * W + 0.08 * W * np.sin(5 * np.arange(H) / H)  # stripe centre, left view
        colour = np.array([140.0, 255.0, 140.0], np.float32)    # BGR, centre of the HSV window

        def paint(img, centre):
            a = np.clip(3.0 * np.exp(-(xs - centre[:, None]) ** 2 / (2 * 2.5 ** 2)), 0, 1)[..., None]
            return img * (1 - a) + colour * a

        left = paint(left, cx)
        dc = d[np.arange(H), np.clip(np.rint(cx).astype(int), 0, W - 1)]
        right = paint(right, cx - dc)
    return np.rint(left).astype(np.uint8), np.rint(right).astype(np.uint8)


def plane_stripe_pair(W, H, D, plane, scale=1.0, seed=0, baseline=0.06):
    """A pair whose laser stripe lies on `plane` (a x + b y + c z + d = 0 in the left camera frame of
    camera_model(W, H, baseline)), on the scene of disparity scale * disparity_field(W, H, D).
    Returns (left_bgr, right_bgr, centres): centres[y] is the true left-view stripe centre of row y (float64; NaN where
    the plane does not cross the row), found by bisection on the analytic disparity field; the right view's stripe is
    painted at x - d(x, y)."""
    rng = np.random.default_rng(seed)
    pad = int(D * 1.5) + 16
    tex = rng.integers(0, 256, (H, W + 2 * pad, 3)).astype(np.float32)
    tex = cv2.GaussianBlur(tex, (0, 0), 1.5)
    tex = np.clip((tex - 128.0) * 2.2 + 110.0, 0, 200)
    di = np.rint(scale * disparity_field(W, H, D)).astype(np.int64)
    xs = np.arange(W)[None, :]
    ys = np.arange(H)[:, None]
    left = tex[ys, xs + pad].copy()
    right = tex[ys, xs + pad + di].copy()
    f = 0.8 * W
    pl = np.asarray(plane, np.float64)
    y = np.arange(H, dtype=np.float64)

    def disp(x):
        return scale * (0.35 * D + 0.20 * D * np.sin(6 * x / W) * np.cos(4 * y / H))

    def g(x):  # the plane's residual at the scene point seen at (x, y), every row at once
        Z = f * baseline / disp(x)
        return pl[0] * (x - W / 2.0) * Z / f + pl[1] * (y - H / 2.0) * Z / f + pl[2] * Z + pl[3]

    lo, hi = np.zeros(H), np.full(H, W - 1.0)
    crosses = g(lo) * g(hi) <= 0
    for _ in range(60):
        m = 0.5 * (lo + hi)
        left_half = g(lo) * g(m) <= 0
        hi = np.where(left_half, m, hi)
        lo = np.where(left_half, lo, m)
    centres = np.where(crosses, 0.5 * (lo + hi), np.nan)
    colour = np.array([140.0, 255.0, 140.0], np.float32)

    def paint(img, centre):
        c = np.where(np.isnan(centre), -1e9, centre)
        a = np.clip(3.0 * np.exp(-(xs - c[:, None]) ** 2 / (2 * 2.5 ** 2)), 0, 1)[..., None]
        return img * (1 - a) + colour * a

    left = paint(left, centres)
    right = paint(right, centres - disp(np.where(crosses, centres, 0.0)))
    return np.rint(left).astype(np.uint8), np.rint(right).astype(np.uint8), centres


def camera_model(W, H, baseline=0.06):
    """K (3x3) and Q (4x4) of the synthetic rig: f = 0.8 W, principal point at the centre."""
    f = 0.8 * W
    K = np.array([[f, 0, W / 2.0], [0, f, H / 2.0], [0, 0, 1]], np.float64)
    Q = np.array([[1, 0, 0, -W / 2.0], [0, 1, 0, -H / 2.0], [0, 0, 0, f], [0, 0, 1.0 / baseline, 0]], np.float64)
    return K, Q


def warp_maps(W, H, seed=0, amplitude=3.0):
    """Identity + smooth +-amplitude px lens-like warp (CV_32FC1 map pair per eye)."""
    xs, ys = np.meshgrid(np.arange(W, dtype=np.float64), np.arange(H, dtype=np.float64))
    u, v = (xs - W / 2) / (W / 2), (ys - H / 2) / (H / 2)
    r2 = u * u + v * v
    ph = 0.7 * seed
    mx = xs + amplitude * (0.6 * u * r2 + 0.4 * np.sin(3 * v + ph))
    my = ys + amplitude * (0.6 * v * r2 + 0.4 * np.cos(3 * u + ph))
    return mx.astype(np.float32), my.astype(np.float32)


LASER_PLANE = np.array([0.3, 0.0, -1.0, 0.4], np.float64)  # default [0,0,1,0] yields all-zero points
