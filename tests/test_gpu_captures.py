"""The frame pipeline on stereo captures as cap.read() delivers them (l3d_pipeline_run_captures_host / _dev): the views
are read in place as strided rows of each capture, and every output must be bit-identical to the pipeline run on the
same views split on the host.  process_frames(frames=...) on top of it, in chunks, against per-frame process_frame."""
import ctypes as C
import json

import numpy as np
import pytest

from laser_3d_reconstruction_b200 import _native as N
from laser_3d_reconstruction_b200 import pipeline, synth
from laser_3d_reconstruction_b200 import system as system_mod

pytestmark = pytest.mark.gpu

KEYS = ("left_rect", "depth", "disp16", "points_2d", "points_3d")


def captures(L, R, split):
    """(n, H, 2W, 3) side by side (split 0) or (n, 2H, W, 3) one above the other (split 1), C-contiguous"""
    return np.ascontiguousarray(np.concatenate([L, R], axis=2 if split == 0 else 1))


def fetch_all(fp, n):
    return [fp.fetch(i) for i in range(n)]


def same_bits(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


def assert_same(want, got, what):
    assert len(want) == len(got)
    for i, (w, g) in enumerate(zip(want, got)):
        for k in KEYS:
            assert same_bits(w[k], g[k]), "%s: %s of frame %d differs" % (what, k, i)


def c1_frames(n, seed0=0):
    W, H, D = 320, 360, 64
    pairs = [synth.stereo_pair(W, H, D, seed=seed0 + s) for s in range(n)]
    return np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])


@pytest.fixture(scope="module")
def c1_data():
    W, H = 320, 360
    K, Q = synth.camera_model(W, H)
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    L, R = c1_frames(16, seed0=40)
    return K, Q, maps, L, R


def check_forms(fp, L, R, what):
    """run_host / run_dev on the split views against run_captures_host / _dev on the captures of both split modes"""
    n = L.shape[0]
    counts = fp.run_host(L, R)
    want = fetch_all(fp, n)
    for split in (0, 1):
        cap = captures(L, R, split)
        assert list(fp.run_captures_host(cap, split)) == list(counts)
        assert_same(want, fetch_all(fp, n), "%s host split %d" % (what, split))
    dl, dr = fp.upload(L), fp.upload(R)
    assert list(fp.run_dev(dl, dr, n)) == list(counts)
    assert_same(want, fetch_all(fp, n), "%s run_dev" % what)
    for split in (0, 1):
        dc = fp.upload(captures(L, R, split))
        assert list(fp.run_captures_dev(dc, n, split)) == list(counts)
        assert_same(want, fetch_all(fp, n), "%s dev split %d" % (what, split))


@pytest.mark.parametrize("lanes", [1, 3, 7, 14])
@pytest.mark.parametrize("use_maps", [True, False])
@pytest.mark.parametrize("use_wls", [True, False])
@pytest.mark.parametrize("mode", [0, 1, 2, 3])
def test_captures_equal_split_views_c1(ctx, c1_data, mode, use_wls, use_maps, lanes):
    """c1 geometry (320x360, 64 disparities, block 5) in every SGBM mode, with and without WLS and rectification maps,
    lane per frame and grouped (7 lanes with WLS and 14 without run the cluster-fused aggregation in modes 0 / 1)"""
    K, Q, maps, L, R = c1_data
    cfg = pipeline.make_pipeline_config(320, 360, 64, 5, mode, Q, K, extractor=N.STEGER_IMPROVED, lanes=lanes,
                                        max_points=8000, use_wls=use_wls, use_maps=use_maps)
    fp = pipeline.FramePipeline(cfg, maps=maps if use_maps else None, ctx=ctx)
    try:
        check_forms(fp, L, R, "mode %d wls %d maps %d lanes %d" % (mode, use_wls, use_maps, lanes))
    finally:
        fp.close()


def test_captures_equal_split_views_c3(ctx):
    """one c3-size case: 1280x720, 128 disparities, block 9, MODE_HH + WLS, grouped over 7 lanes"""
    W, H, D, bs = 1280, 720, 128, 9
    K, Q = synth.camera_model(W, H)
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    pairs = [synth.stereo_pair(W, H, D, seed=70 + s) for s in range(3)]
    L, R = np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])
    cfg = pipeline.make_pipeline_config(W, H, D, bs, 1, Q, K, extractor=N.STEGER_IMPROVED, lanes=7, max_points=20000)
    fp = pipeline.FramePipeline(cfg, maps=maps, ctx=ctx)
    try:
        check_forms(fp, L, R, "c3")
    finally:
        fp.close()


def test_captures_graph_replay_keeps_input_forms_apart(ctx, c1_data):
    """A repeated launch-bound c1 host step is replayed as a CUDA graph.  Steps on split views and on captures of both
    split modes alternate on one pipeline (the two capture forms even share one pinned buffer, rewritten in place):
    every step, replayed or not, gives the results of the split views."""
    K, Q, maps, L, R = c1_data
    n = 14
    L, R = L[:n], R[:n]
    cfg = pipeline.make_pipeline_config(320, 360, 64, 5, 1, Q, K, extractor=N.STEGER_IMPROVED, lanes=14, max_points=8000)
    fp = pipeline.FramePipeline(cfg, maps=maps, ctx=ctx)
    try:
        pL = pipeline.pinned_empty(L.shape, np.uint8); pR = pipeline.pinned_empty(R.shape, np.uint8)
        pL[:] = L; pR[:] = R
        pC = pipeline.pinned_empty((n * 2 * 360 * 320 * 3,), np.uint8)  # the bytes of either capture form
        fp.run_host(pL, pR)
        want = fetch_all(fp, n)
        replays = {}
        for it in range(6):
            before = fp.graph_replays
            fp.run_host(pL, pR)
            assert_same(want, fetch_all(fp, n), "split views, step %d" % it)
            replays["eyes"] = replays.get("eyes", 0) + fp.graph_replays - before
            for split in (0, 1):
                cap = captures(L, R, split)
                c = pC.reshape(cap.shape)
                c[:] = cap
                before = fp.graph_replays
                fp.run_captures_host(c, split)
                assert_same(want, fetch_all(fp, n), "captures split %d, step %d" % (split, it))
                replays[split] = replays.get(split, 0) + fp.graph_replays - before
        assert fp.graph_replays > 0
        assert replays["eyes"] > 0 and replays[0] > 0 and replays[1] > 0, replays
    finally:
        fp.close()


def test_captures_refuse_bad_arguments(ctx):
    W, H = 64, 32
    K, Q = synth.camera_model(W, H)
    cfg = pipeline.make_pipeline_config(W, H, 16, 3, 2, Q, K, lanes=1, max_points=64, use_wls=False, use_maps=False)
    fp = pipeline.FramePipeline(cfg, ctx=ctx)
    try:
        good0 = np.zeros((2, H, 2 * W, 3), np.uint8)
        good1 = np.zeros((2, 2 * H, W, 3), np.uint8)
        for bad, split in ((good1, 0), (good0, 1), (good0.astype(np.int16), 0), (good0[:, :, ::2], 0),
                           (np.zeros((2, H, 2 * W + 2, 3), np.uint8), 0), (good0[0], 0), (good0[:0], 0), (good0, 2)):
            with pytest.raises(N.L3DError):
                fp.run_captures_host(bad, split)
        with pytest.raises(N.L3DError):
            fp.run_captures_dev(1, 2, 2)
        counts = (C.c_int * 2)()
        p = C.c_void_p(good0.ctypes.data)
        lib = fp.lib  # L3D_ERR_ARG = -1
        for split in (-1, 2, 7):
            assert lib.l3d_pipeline_run_captures_host(fp.h, p, 2, split, None, None, counts) == -1
            assert lib.l3d_pipeline_run_captures_dev(fp.h, p, 2, split, counts) == -1
        assert lib.l3d_pipeline_run_captures_host(fp.h, None, 2, 0, None, None, counts) == -1
        assert lib.l3d_pipeline_run_captures_host(fp.h, p, 0, 0, None, None, counts) == -1
        assert lib.l3d_pipeline_run_captures_dev(fp.h, None, 2, 0, counts) == -1
        assert lib.l3d_pipeline_run_captures_dev(fp.h, p, -1, 1, counts) == -1
        # the refusals left the pipeline usable
        assert len(fp.run_captures_host(good0, 0)) == 2
    finally:
        fp.close()


# ---- process_frames(frames=...) --------------------------------------------------------------------------------------
class _FakeCapture:
    def __init__(self, frames):
        self.frames, self.i = list(frames), 0

    def isOpened(self):
        return True

    def read(self):
        if self.i >= len(self.frames):
            return False, None
        self.i += 1
        return True, self.frames[self.i - 1]

    def release(self):
        pass


def _calibration(tmp_path, W, H, dist=True):
    K, _ = synth.camera_model(W, H)
    d = ([[0.01, -0.02, 0.0, 0.0, 0.0]], [[-0.01, 0.015, 0.0, 0.0, 0.0]]) if dist else ([[0.0] * 5], [[0.0] * 5])
    calib = dict(R=np.eye(3).tolist(), T=[[-0.06], [0.0], [0.0]], camera_matrix_left=K.tolist(), dist_coeffs_left=d[0],
                 camera_matrix_right=K.tolist(), dist_coeffs_right=d[1])
    path = tmp_path / "stereo_calibration.json"
    path.write_text(json.dumps(calib))
    return str(path)


def _system(path, W, H, split_mode, cfg):
    import laser_3d_reconstruction_b200 as l3d
    from laser_3d_reconstruction_b200.system import LaserReconstructionSystem
    w, h = (2 * W, H) if split_mode == 'horizontal' else (W, 2 * H)
    cam = l3d.SingleUSBStereoCameraManager(width=w, height=h, split_mode=split_mode, calibration_file=path, verbose=False)
    assert cam.initialize_offline()
    s = LaserReconstructionSystem(cfg, verbose=False)
    assert s.initialize(camera=cam)
    return s, cam


def _per_frame(path, W, H, split_mode, cfg, caps):
    s, cam = _system(path, W, H, split_mode, cfg)
    cam.cap = _FakeCapture(caps)
    got = [s.process_frame() for _ in range(len(caps))]
    return s, got


def _assert_batched_equal(got, out, sysA, sysB, want_images, elem_type):
    assert len(out) == len(got) and sysB.frame_count == sysA.frame_count == len(got)
    for i, ((g_rect, g_depth, g_pts), (b_rect, b_depth, b_pts)) in enumerate(zip(got, out)):
        if want_images:
            assert b_rect.dtype == np.uint8 and b_depth.dtype == np.float32 and b_rect.flags.owndata and b_depth.flags.owndata
            assert same_bits(b_rect, g_rect) and same_bits(b_depth, g_depth), "frame %d images" % i
        else:
            assert b_rect is None and b_depth is None
        assert b_pts == g_pts, "frame %d points" % i
        assert all(type(x) is elem_type and type(y) is elem_type for x, y in b_pts)
    assert sysB.point_cloud == sysA.point_cloud


@pytest.mark.parametrize("split_mode", ["horizontal", "vertical"])
def test_process_frames_captures_in_chunks(tmp_path, split_mode):
    """More frames than two chunks, as one capture array, as a list and without images: exactly the per-frame results"""
    import laser_3d_reconstruction_b200 as l3d
    W, H, D = 320, 360, 64
    n = 2 * system_mod.CHUNK_FRAMES + 3
    base = [synth.stereo_pair(W, H, D, seed=s) for s in range(8)]
    caps = []
    for i in range(n):
        l, r = base[i % len(base)][0].copy(), base[(i + i // len(base)) % len(base)][1].copy()
        l[:4, :4] = i % 251  # every frame distinct
        caps.append(np.concatenate([l, r], axis=1 if split_mode == 'horizontal' else 0))
    path = _calibration(tmp_path, W, H)
    cfg = l3d.Config()
    sysA, got = _per_frame(path, W, H, split_mode, cfg, caps)
    assert sum(len(g[2]) for g in got) > 0 and len(sysA.point_cloud) > 0
    arr = np.stack(caps)
    for frames, want_images in ((arr, True), (list(caps), True), (arr, False)):
        sysB, _ = _system(path, W, H, split_mode, cfg)
        out = sysB.process_frames(frames=frames, lanes=3, want_images=want_images)
        _assert_batched_equal(got, out, sysA, sysB, want_images, np.float64)
        sysB.stop()
    sysA.stop()


def test_process_frames_chunk_overflow_reruns_that_chunk_only(tmp_path, monkeypatch):
    """FastSteger on a bright noisy patch in one frame of the middle chunk overflows the point lists: that chunk alone
    runs again on a larger pipeline; the chunks before it are not accumulated twice."""
    import laser_3d_reconstruction_b200 as l3d
    W, H, D = 640, 480, 64
    monkeypatch.setattr(system_mod, "CHUNK_FRAMES", 2)
    pairs = [synth.stereo_pair(W, H, D, seed=s) for s in range(5)]
    pairs[3][0][20:460, 20:620] = np.random.default_rng(5).integers(235, 256, (440, 600, 1), dtype=np.uint8)
    caps = [np.ascontiguousarray(np.concatenate([l, r], axis=1)) for l, r in pairs]
    path = _calibration(tmp_path, W, H, dist=False)
    cfg = l3d.Config()
    cfg.LASER_EXTRACTOR_TYPE = 'steger'
    sysA, got = _per_frame(path, W, H, 'horizontal', cfg, caps)
    assert len(got[3][2]) > 20000 and max(len(g[2]) for i, g in enumerate(got) if i != 3) <= 20000
    runs = []
    orig = pipeline.FramePipeline.run_captures_host

    def counted(self, frames, split, *a, **k):
        runs.append((frames.shape[0], self.cfg.max_points))
        return orig(self, frames, split, *a, **k)

    monkeypatch.setattr(pipeline.FramePipeline, "run_captures_host", counted)
    sysB, _ = _system(path, W, H, 'horizontal', cfg)
    out = sysB.process_frames(frames=np.stack(caps), lanes=2)
    assert [r[0] for r in runs] == [2, 2, 2, 1] and runs[0][1] == runs[1][1] < runs[2][1] == runs[3][1]
    _assert_batched_equal(got, out, sysA, sysB, True, np.float32)
    sysA.stop(); sysB.stop()
