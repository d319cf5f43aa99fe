import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


# scripts, not test modules: the differential fuzzers and the verbose bring-up checkers are run by hand
collect_ignore_glob = ["fuzz/*", "bringup/*"]


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden_synth():
    return dict(np.load(os.path.join(GOLDEN, "synth_c1.npz")))


def _load_golden(*names):
    """one dict of every array in tests/golden/<name>.npz (the real pairs are stored one per file)"""
    out = {}
    for n in names:
        out.update(np.load(os.path.join(GOLDEN, n + ".npz")))
    return out


@pytest.fixture(scope="session")
def golden_real():
    """the shipped calibration of the real rig and two of its pairs (a, b) in full"""
    return _load_golden("real_rig", "real_pair_a", "real_pair_b")


@pytest.fixture(scope="session")
def golden_real_more():
    """four more real pairs (c-f): inputs, int16 disparity, CRC32s of the rectified views and the depth image"""
    return _load_golden("real_pair_c", "real_pair_d", "real_pair_e", "real_pair_f")


@pytest.fixture(scope="session")
def ctx():
    """One GPU context for the whole session; fails loudly when no GPU / library is present."""
    from laser_3d_reconstruction_b200 import _native
    c = _native.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="session")
def rect_cases(golden_real):
    """(K, dist, R, P, size) sets for the rectification-map tests: the real rig at two sizes + a synthetic 12-coefficient rig."""
    import cv2
    g = golden_real
    cases = []
    for size in ((320, 240), (640, 480)):
        K1, d1, K2, d2 = g["K_left"], g["dist_left"], g["K_right"], g["dist_right"]
        s = size[0] / 320.0
        S = np.diag([s, s, 1.0])
        R1, R2, P1, P2, Q, _, _ = cv2.stereoRectify(S @ K1, d1, S @ K2, d2, size, g["R"], g["T"], alpha=0)
        cases += [(S @ K1, d1, R1, P1, size), (S @ K2, d2, R2, P2, size)]
    # synthetic rig with 8 distortion coefficients + thin prism terms
    K = np.array([[1024.0, 0, 655.3], [0, 1019.5, 349.2], [0, 0, 1]])
    d = np.array([-0.21, 0.09, 0.0012, -0.0007, -0.015, 0.02, -0.01, 0.003, 0.0004, -0.0002, 0.0003, 0.0001])
    Rr = cv2.Rodrigues(np.array([0.01, -0.02, 0.005]))[0]
    P = np.array([[980.0, 0, 640.0, 0], [0, 980.0, 360.0, 0], [0, 0, 1, 0]])
    cases.append((K, d, Rr, P, (1280, 720)))
    return cases
