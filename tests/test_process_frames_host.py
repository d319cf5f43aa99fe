"""CPU-side checks of the capture entry points of the frame pipeline: the Python shape checks of run_captures_host, and
the chunk bookkeeping of LaserReconstructionSystem.process_frames against a stand-in pipeline (no GPU needed)."""
import types

import numpy as np
import pytest

from laser_3d_reconstruction_b200 import _native as N
from laser_3d_reconstruction_b200 import pipeline
from laser_3d_reconstruction_b200 import system as system_mod


class _NoLib:
    def __getattr__(self, name):
        raise AssertionError("%s called although the arguments are invalid" % name)


def _pipe_without_device(W=8, H=4):
    fp = pipeline.FramePipeline.__new__(pipeline.FramePipeline)
    fp.cfg = pipeline.make_pipeline_config(W, H, 16, 3, 1, None, np.eye(3), lanes=1, max_points=16)
    fp.lib = _NoLib()
    return fp


def test_run_captures_host_refuses_wrong_shapes_before_any_native_call():
    fp = _pipe_without_device(W=8, H=4)
    assert fp.capture_shape(5, 0) == (5, 4, 16, 3) and fp.capture_shape(5, 1) == (5, 8, 8, 3)
    side = np.zeros((2, 4, 16, 3), np.uint8)
    top = np.zeros((2, 8, 8, 3), np.uint8)
    for bad, split in ((top, 0), (side, 1), (side.astype(np.float32), 0), (side[:, :, ::-1], 0), (side[0], 0),
                       (side[:0], 0), (np.zeros((2, 4, 17, 3), np.uint8), 0), (np.zeros((2, 4, 16, 4), np.uint8), 0),
                       (side, 2), (side, -1), (side, None)):
        with pytest.raises(N.L3DError):
            fp.run_captures_host(bad, split)
    with pytest.raises(N.L3DError):
        fp.run_captures_host(side, 0, depth_out=np.zeros((1, 4, 8), np.float32))
    with pytest.raises(N.L3DError):
        fp.run_captures_dev(0, 2, 3)


def test_points_to_list_f64_gives_what_row_unpacking_gives():
    a = np.random.default_rng(3).random((50, 2))
    got = N.points_to_list_f64(a)
    assert got == [(x, y) for x, y in a]
    assert all(type(x) is np.float64 and type(y) is np.float64 for x, y in got)
    assert N.points_to_list_f64(np.empty((0, 2))) == []


class _StandIn:
    """A frame pipeline whose 'frames' carry their number in pixel (0, 0, 0) and a point-count demand in (0, 0, 1)
    (x 1000).  Each frame yields the 2D point (id, id + 0.5) and the 3D rows (id, 0, 0) and a NaN row."""

    def __init__(self, W, H, cap, extractor, log):
        self.cfg = types.SimpleNamespace(W=W, H=H, max_points=cap, extractor=extractor)
        self.log, self.ids, self.need = log, [], 0

    def _run(self, ids, demand, form):
        self.log.append((form, list(ids), self.cfg.max_points))
        self.ids = [int(i) for i in ids]
        self.need = int(max(demand)) * 1000
        return np.ones(len(ids), np.int32)

    def run_captures_host(self, frames, split):
        assert frames.flags.c_contiguous and frames.dtype == np.uint8
        return self._run(frames[:, 0, 0, 0], frames[:, 0, 0, 1], ("captures", split))

    def run_host(self, left, right):
        return self._run(left[:, 0, 0, 0], left[:, 0, 0, 1], "eyes")

    @property
    def points_needed(self):
        return self.need

    def fetch_points(self, i, want_2d=False):
        f = self.ids[i]
        return np.array([[f, f + 0.5]]), np.array([[f, 0.0, 0.0], [np.nan, 1.0, 1.0]])

    def fetch_images(self, i):
        f = self.ids[i]
        return np.full((self.cfg.H, self.cfg.W, 3), f, np.uint8), np.full((self.cfg.H, self.cfg.W), f, np.float32)


def _system(monkeypatch, split_mode, extractor, chunk=4):
    monkeypatch.setattr(system_mod, "CHUNK_FRAMES", chunk)
    s = system_mod.LaserReconstructionSystem(verbose=False)
    s.camera = types.SimpleNamespace(split_mode=split_mode)
    log = []
    s._pipeline = lambda lanes, cap=None: _StandIn(400, 300, max(20000, int(cap or 0)), extractor, log)
    return s, log


def _captures(n, split_mode, big=()):
    shape = (n, 4, 16, 3) if split_mode == 'horizontal' else (n, 8, 8, 3)
    a = np.zeros(shape, np.uint8)
    a[:, 0, 0, 0] = np.arange(n)
    a[:, 0, 0, 1] = 1
    for i in big:
        a[i, 0, 0, 1] = 30  # 30 000 points: more than the default capacity
    return a


@pytest.mark.parametrize("split_mode,split", [("horizontal", 0), ("vertical", 1)])
def test_process_frames_runs_captures_in_chunks(monkeypatch, split_mode, split):
    s, log = _system(monkeypatch, split_mode, N.EXTRACT_SIMPLE)
    a = _captures(11, split_mode)
    out = s.process_frames(frames=a)
    assert log == [(("captures", split), [0, 1, 2, 3], 20000), (("captures", split), [4, 5, 6, 7], 20000),
                   (("captures", split), [8, 9, 10], 20000)]
    assert [o[2] for o in out] == [[(np.float64(f), np.float64(f + 0.5))] for f in range(11)]
    assert all(type(o[2][0][0]) is np.float64 for o in out)
    assert [int(o[0][0, 0, 0]) for o in out] == list(range(11)) and all(o[1][0, 0] == f for f, o in enumerate(out))
    assert s.point_cloud == [[float(f), 0.0, 0.0] for f in range(11)] and s.frame_count == 11
    # a list, and any other iterable, of captures: stacked one chunk at a time, same results
    for frames in (list(a), (f for f in a)):
        s2, log2 = _system(monkeypatch, split_mode, N.EXTRACT_SIMPLE)
        out2 = s2.process_frames(frames=frames, want_images=False)
        assert log2 == log and [o[2] for o in out2] == [o[2] for o in out]
        assert all(o[0] is None and o[1] is None for o in out2) and s2.point_cloud == s.point_cloud
    # split views keep their own entry point, in chunks too
    s3, log3 = _system(monkeypatch, split_mode, N.STEGER_FAST)
    eyes = np.zeros((6, 4, 8, 3), np.uint8)
    eyes[:, 0, 0, 0] = np.arange(6)
    eyes[:, 0, 0, 1] = 1
    out3 = s3.process_frames(lefts=eyes, rights=eyes)
    assert [e[1] for e in log3] == [[0, 1, 2, 3], [4, 5]] and all(e[0] == "eyes" for e in log3)
    assert all(type(o[2][0][0]) is np.float32 for o in out3)


def test_process_frames_overflowing_chunk_runs_again_alone(monkeypatch):
    s, log = _system(monkeypatch, "horizontal", N.STEGER_FAST)
    out = s.process_frames(frames=_captures(10, "horizontal", big=(5,)))
    assert [(e[1], e[2]) for e in log] == [([0, 1, 2, 3], 20000), ([4, 5, 6, 7], 20000), ([4, 5, 6, 7], 60000),
                                           ([8, 9], 60000)]
    assert s.point_cloud == [[float(f), 0.0, 0.0] for f in range(10)] and s.frame_count == 10 and len(out) == 10
    # a demand beyond even the grown capacity (W * H bounds it) is an error, not a silent truncation
    s2, _ = _system(monkeypatch, "horizontal", N.STEGER_FAST)
    monkeypatch.setattr(_StandIn, "points_needed", property(lambda self: self.cfg.max_points + 1))
    with pytest.raises(N.L3DError):
        s2.process_frames(frames=_captures(3, "horizontal"))
    assert s2.point_cloud == [] and s2.frame_count == 0
