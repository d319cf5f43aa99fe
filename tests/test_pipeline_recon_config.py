"""Host-side configuration of the frame pipeline's reconstruction: the ReconParams make_pipeline_config stores for each kind,
and the left matcher depth_config runs without the WLS filter (as constructed, or as createDisparityWLSFilter mutates it)."""
import numpy as np
import pytest

from laser_3d_reconstruction_b200 import _native as N
from laser_3d_reconstruction_b200 import pipeline, synth
from laser_3d_reconstruction_b200.improved_reconstruction import ImprovedLaserReconstructor
from oracle import ref_ops

W, H, D, BS = 320, 360, 64, 5


def fields(s):
    return {k: (list(getattr(s, k)) if hasattr(getattr(s, k), "__len__") else getattr(s, k)) for k, _ in s._fields_}


def test_default_recon_is_depth_with_K():
    K, Q = synth.camera_model(W, H)
    cfg = pipeline.make_pipeline_config(W, H, D, BS, 2, Q, K)
    want = N.ReconParams()
    want.kind = N.RECON_DEPTH
    want.K[:] = list(K.reshape(9))
    want.n_water = 1.33
    assert fields(cfg.recon) == fields(want)


@pytest.mark.parametrize("kind,window,min_disparity", [(N.RECON_DISPARITY, 3, 1.0), (N.RECON_DISPARITY_MEDIAN, 1, 1.0),
                                                       (N.RECON_DISPARITY_MEDIAN, 5, 22.5), (N.RECON_DISPARITY_MEDIAN, 9, 0.0)])
def test_disparity_kinds_from_the_reconstructor(kind, window, min_disparity):
    K, Q = synth.camera_model(W, H, baseline=0.8)
    ir = ImprovedLaserReconstructor(Q, verbose=False)
    cfg = pipeline.make_pipeline_config(W, H, D, BS, 1, Q, K, recon=ir.recon_params(kind, min_disparity, window))
    r = cfg.recon
    ref = ref_ops.ImprovedLaserReconstructorRef(Q)
    assert (r.kind, r.window, r.min_disparity) == (kind, window, min_disparity)
    assert (r.fx, r.baseline, r.cx, r.cy) == (ref.fx, ref.baseline, ref.cx, ref.cy) == (0.8 * W, 0.8, W / 2.0, H / 2.0)
    # the depth path is the default one: both matchers and the WLS filter
    assert cfg.depth.use_wls == 1 and fields(cfg.depth.left) == fields(pipeline.wls_mutate(pipeline.sgbm_params(D, BS, 1)))


@pytest.mark.parametrize("mode", [0, 1, 2, 3])
def test_left_matcher_without_wls(mode):
    K, Q = synth.camera_model(W, H)
    base, mutated, _ = ref_ops.sgbm_param_sets(D, BS, mode)
    as_constructed = pipeline.depth_config(D, BS, mode, Q, use_wls=False)
    assert as_constructed.use_wls == 0 and fields(as_constructed.left) == base
    m = pipeline.depth_config(D, BS, mode, Q, use_wls=False, mutated_left=True)
    assert m.use_wls == 0 and fields(m.left) == mutated
    assert fields(pipeline.depth_config(D, BS, mode, Q, use_wls=True, mutated_left=True).left) == mutated
    cfg = pipeline.make_pipeline_config(W, H, D, BS, mode, Q, K, use_wls=False, mutated_left=True)
    assert cfg.depth.use_wls == 0 and fields(cfg.depth.left) == mutated
    assert fields(pipeline.make_pipeline_config(W, H, D, BS, mode, Q, K, use_wls=False).depth.left) == base
