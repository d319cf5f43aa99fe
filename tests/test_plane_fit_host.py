"""CPU-side checks of the laser-plane fit: the hypothesis index generator, the numpy restatement (oracle/plane_fit.py),
the ctypes structs of l3d_fit_plane, the synthetic plane-stripe renderer and calibrate_laser_plane's host logic."""
import ctypes as C
import hashlib
import types

import numpy as np
import pytest

from laser_3d_reconstruction_b200 import _native as N
from laser_3d_reconstruction_b200 import synth
from laser_3d_reconstruction_b200 import system as system_mod
from oracle import plane_fit as opf


def test_hypothesis_indices_hand_checked():
    # seed 0: z = (3h + k + 1) * 0x9E3779B97F4A7C15 is the splitmix64 state sequence from 0, whose first outputs are the
    # published ones
    want = [0xE220A8397B1DCDAF, 0x6E789E6AA1B965F4, 0x06C45D188009454F]
    assert [int(v) for v in opf.splitmix64(np.array([(j * opf.GOLDEN) & opf.M64 for j in (1, 2, 3)], np.uint64))] == want
    n = 1000003
    assert opf.hypothesis_indices(n, 1, 0).tolist() == [[w % n for w in want]]

    def one(seed, h, k, n):  # plain Python integers
        z = (seed + (3 * h + k + 1) * opf.GOLDEN) & opf.M64
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & opf.M64
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & opf.M64
        return (z ^ (z >> 31)) % n

    for seed in (0, 1, 12345, 2 ** 64 - 1):
        for n in (3, 7, 200003):
            got = opf.hypothesis_indices(n, 50, seed)
            assert got.tolist() == [[one(seed, h, k, n) for k in range(3)] for h in range(50)]


def _plane_cloud(n, outliers, sigma, seed, plane=(0.3, -0.2, 0.9, 0.7)):
    rng = np.random.default_rng(seed)
    pl = np.asarray(plane, np.float64)
    pl = pl / np.linalg.norm(pl[:3])
    a = np.cross(pl[:3], [1.0, 0, 0]); a /= np.linalg.norm(a)
    b = np.cross(pl[:3], a)
    uv = rng.uniform(-0.5, 0.5, (n, 2))
    pts = -pl[3] * pl[:3] + uv[:, :1] * a + uv[:, 1:] * b + sigma * rng.standard_normal((n, 1)) * pl[:3]
    k = int(outliers * n)
    pts[:k] = rng.uniform(-1, 1, (k, 3)) + [0, 0, 1]
    return pts, pl


def test_oracle_recovers_planes():
    for seed in range(3):
        pts, pl = _plane_cloud(3000, 0.4, 0.0, seed)
        r = opf.fit_plane(pts, 1e-3, 256, seed)
        assert np.abs(r["plane"] - pl).max() < 1e-12 and r["inliers"] >= 1800 and r["rms"] < 1e-12
        pts, pl = _plane_cloud(3000, 0.3, 3e-4, seed)
        r = opf.fit_plane(pts, 1.5e-3, 256, seed)
        assert np.degrees(np.arccos(min(1.0, r["plane"][:3] @ pl[:3]))) < 0.1 and abs(r["plane"][3] - pl[3]) < 1e-4
        assert r["eig"][0] < r["eig"][1] <= r["eig"][2] and 1 <= r["refits"] <= 10
    # RANSAC counts: invalid hypotheses (a repeated or non-finite point) are -1 and never win
    pts = np.array([[0.0, 0, 0], [1, 0, 0], [0, 1, 0], [np.nan, 0, 0]])
    win, cnt, counts = opf.ransac(pts, 0.1, 64, 0)
    assert counts.min() == -1 and cnt == 3 and counts[win] == 3 and (counts[:win] < 3).all()


def test_plane_fit_structs_match_header():
    assert C.sizeof(N.PlaneFitParams) == 24 and N.PlaneFitParams.seed.offset == 16
    assert C.sizeof(N.PlaneFitResult) == 88
    assert (N.PlaneFitResult.inliers.offset, N.PlaneFitResult.rms.offset, N.PlaneFitResult.eig.offset,
            N.PlaneFitResult.hypothesis.offset, N.PlaneFitResult.hypothesis_inliers.offset,
            N.PlaneFitResult.refits.offset) == (32, 40, 48, 72, 76, 80)


def test_plane_stripe_pair_centres_lie_on_the_plane():
    W, H, D = 320, 360, 64
    f, B = 0.8 * W, 0.06
    plane = np.array([0.89, -0.09, 0.445, -0.336])
    for scale in (0.75, 1.0, 1.25):
        L, R, c = synth.plane_stripe_pair(W, H, D, plane, scale, seed=1)
        assert L.shape == R.shape == (H, W, 3) and L.dtype == np.uint8 and c.shape == (H,)
        ok = ~np.isnan(c)
        assert ok.sum() > 300
        y, x = np.arange(H)[ok], c[ok]
        Z = f * B / (scale * (0.35 * D + 0.20 * D * np.sin(6 * x / W) * np.cos(4 * y / H)))
        P = np.stack([(x - W / 2) * Z / f, (y - H / 2) * Z / f, Z], 1)
        assert np.abs(P @ plane[:3] + plane[3]).max() < 1e-9
        # the stripe is painted at the centre: the middle of each row's saturated run in the left view
        rows = np.nonzero(ok & (c > 8) & (c < W - 9))[0]
        sat = L[rows, :, 1] == 255
        mid = (sat * np.arange(W)).sum(1) / sat.sum(1)
        assert np.abs(mid - c[rows]).max() <= 0.6
    _, _, c = synth.plane_stripe_pair(W, H, D, [0.0, 0.0, 1.0, 100.0], 1.0)  # Z = -100: crosses no row
    assert np.isnan(c).all()


def test_existing_synth_outputs_unchanged():
    h = hashlib.sha256()
    for a in (synth.stereo_pair(320, 360, 64, seed=0) + synth.stereo_pair(96, 40, 16, seed=3, laser=False)
              + synth.camera_model(320, 360) + synth.warp_maps(64, 48, 1) + (synth.disparity_field(64, 48, 16), synth.LASER_PLANE)):
        h.update(a.tobytes())
    assert h.hexdigest() == "04e2e62cb10adab3638bdccedba62207b5ce55d89f7b17e58c140ff24d4c0772"


class _StandIn:
    """frames carry their number in pixel (0, 0, 0); each yields one 3D point (id, 0, 1)"""

    def __init__(self, cap, log):
        self.cfg = types.SimpleNamespace(W=400, H=300, max_points=cap)
        self.log, self.ids = log, []

    def run_captures_host(self, frames, split):
        self.ids = [int(i) for i in frames[:, 0, 0, 0]]
        self.log.append(("captures", split, self.ids))
        return np.ones(len(self.ids), np.int32)

    def run_host(self, left, right):
        self.ids = [int(i) for i in left[:, 0, 0, 0]]
        self.log.append(("eyes", self.ids))
        return np.ones(len(self.ids), np.int32)

    points_needed = 0

    def fetch_points(self, i, want_2d=False):
        return np.array([[float(self.ids[i]), 0.0, 1.0]])


def test_calibrate_laser_plane_host_logic(monkeypatch):
    from laser_3d_reconstruction_b200.config import Config
    monkeypatch.setattr(system_mod, "CHUNK_FRAMES", 4)
    s = system_mod.LaserReconstructionSystem(verbose=False)
    with pytest.raises(ValueError, match="calibrat"):
        s.calibrate_laser_plane(frames=np.zeros((2, 4, 16, 3), np.uint8))  # no camera
    s.camera = types.SimpleNamespace(split_mode="horizontal", Q=None, device=0)
    with pytest.raises(ValueError, match="calibrat"):
        s.calibrate_laser_plane(frames=np.zeros((2, 4, 16, 3), np.uint8))
    _, Q = synth.camera_model(320, 360)
    s.camera.Q = Q
    s.reconstructor = types.SimpleNamespace(laser_plane=Config.LASER_PLANE_COEFFICIENTS)
    s.point_cloud, s.frame_count = [[1.0, 2.0, 3.0]], 7
    log, recons = [], []

    def pipe(lanes, cap=None, recon=None):
        recons.append((lanes, recon))
        return _StandIn(max(20000, int(cap or 0)), log)

    s._pipeline = pipe
    seen = {}

    def fake_fit(points, threshold, hypotheses, seed, device=0):
        seen.update(points=points, args=(threshold, hypotheses, seed, device))
        return types.SimpleNamespace(plane=np.array([0.0, 0.6, 0.8, 0.5]))

    monkeypatch.setattr(system_mod, "fit_laser_plane", fake_fit)
    frames = np.zeros((10, 4, 16, 3), np.uint8)
    frames[:, 0, 0, 0] = np.arange(10)
    fit = s.calibrate_laser_plane(frames=frames, threshold=0.004, hypotheses=512, seed=9, window=5, min_disparity=2.0, lanes=3)
    assert [e[2] for e in log] == [[0, 1, 2, 3], [4, 5, 6, 7], [8, 9]] and all(e[:2] == ("captures", 0) for e in log)
    assert all(lanes == 3 and r.kind == N.RECON_DISPARITY_MEDIAN and r.window == 5 and r.min_disparity == 2.0
               and r.fx == 256.0 and abs(r.baseline - 0.06) < 1e-15 for lanes, r in recons)
    assert seen["points"].tolist() == [[float(i), 0.0, 1.0] for i in range(10)] and seen["args"] == (0.004, 512, 9, 0)
    assert s.reconstructor.laser_plane.tolist() == [0.0, 0.6, 0.8, 0.5] == s.config.LASER_PLANE_COEFFICIENTS.tolist()
    assert fit.plane.tolist() == [0.0, 0.6, 0.8, 0.5]
    assert Config.LASER_PLANE_COEFFICIENTS.tolist() == [0, 0, 1, 0]  # the class keeps the reference's constant
    assert s.point_cloud == [[1.0, 2.0, 3.0]] and s.frame_count == 7
    # the default threshold follows the camera's depth configuration: 10 mm with the WLS filter, else 5 mm
    for use_wls, want in ((1, 0.01), (0, 0.005)):
        s.camera._depth_config = lambda use_wls=use_wls: types.SimpleNamespace(use_wls=use_wls)
        s.calibrate_laser_plane(frames=frames)
        assert seen["args"][0] == want
    log.clear()
    s.calibrate_laser_plane(lefts=frames[:, :, :8], rights=frames[:, :, 8:])
    assert [e[1] for e in log] == [[0, 1, 2, 3], [4, 5, 6, 7], [8, 9]] and all(e[0] == "eyes" for e in log)


def test_calibrate_laser_plane_without_laser_points(monkeypatch):
    s = system_mod.LaserReconstructionSystem(verbose=False)
    _, Q = synth.camera_model(320, 360)
    s.camera = types.SimpleNamespace(split_mode="horizontal", Q=Q, device=0)
    s._pipeline = lambda lanes, cap=None, recon=None: _NoPoints(max(20000, int(cap or 0)))
    monkeypatch.setattr(system_mod, "fit_laser_plane", lambda *a, **k: pytest.fail("fit called without points"))
    with pytest.raises(ValueError, match="laser line was not detected"):
        s.calibrate_laser_plane(frames=np.zeros((3, 4, 16, 3), np.uint8))


class _NoPoints(_StandIn):
    def __init__(self, cap):
        super().__init__(cap, [])

    def fetch_points(self, i, want_2d=False):
        return np.empty((0, 3))
