"""The wavefront aggregation's paired previous-row paths (sgm_step_pair in csrc/sgm_step.cuh, used by sgbm_vwave_kernel at
D = 128 with an even number of columns per warp): two columns share each 32-bit word, one per 16-bit half.

The CPU tests check the packing identities of the step and a numpy restatement of the whole paired step against the plain
SGM recurrence.  The GPU tests run the frame pipeline in grouped mode on geometries that select 4 to 9 columns per warp,
8-, 9- and 16-CTA clusters, full and partial last strips; each run asserts from the launched kernels' names that the
wavefront kernel ran with the expected columns per warp.  The disparity is compared bit for bit with cv2 (one matcher,
uniquenessRatio 10 and 0) and with the lane-per-frame pipeline, whose direction-split kernels share no code with the
wavefront kernel (WLS: the left and the right matcher)."""
import os

import cv2
import numpy as np
import pytest

from oracle import ref_ops

MASK16 = np.uint32(0xffff)


def prmt(a, b, sel):
    """PRMT / __byte_perm in its default mode: byte i of the result is byte (sel >> 4 i) & 7 of the pair {b:a}."""
    a, b = a.astype(np.uint64), b.astype(np.uint64)
    x = a | (b << np.uint64(32))
    out = np.zeros_like(a)
    for i in range(4):
        s = np.uint64((sel >> (4 * i)) & 7)
        out |= ((x >> (np.uint64(8) * s)) & np.uint64(0xff)) << np.uint64(8 * i)
    return out.astype(np.uint32)


def test_paired_step_packing_identities():
    rng = np.random.default_rng(7)
    lo = rng.integers(0, 1 << 16, (1000, 32), dtype=np.uint32)
    hi = rng.integers(0, 1 << 16, (1000, 32), dtype=np.uint32)
    m = lo | (hi << np.uint32(16))                       # one min-tree result per lane: (min a | min b << 16)
    # two CREDUX.MIN over the warp: on m (high half = min of the high halves) and on m << 16 (high half = min of the lows)
    r_hi = m.min(axis=1)
    r_lo = ((m.astype(np.uint64) << np.uint64(16)) & np.uint64(0xffffffff)).astype(np.uint32).min(axis=1)
    assert np.array_equal(r_hi >> np.uint32(16), hi.min(axis=1))
    assert np.array_equal(r_lo >> np.uint32(16), lo.min(axis=1))
    # PRMT 0x7632 repacks them as (min a | min b << 16), the layout the next step's minI2 expects
    packed = prmt(r_lo, r_hi, 0x7632)
    assert np.array_equal(packed & MASK16, lo.min(axis=1))
    assert np.array_equal(packed >> np.uint32(16), hi.min(axis=1))

    # column interleave of the costs and the way back: word k of lane l = disparity 4l + k of columns (a, b)
    ca = rng.integers(0, 1 << 32, (100, 32, 2), dtype=np.uint64).astype(np.uint32)   # sgm_step layout: 2 words per lane
    cb = rng.integers(0, 1 << 32, (100, 32, 2), dtype=np.uint64).astype(np.uint32)
    w = [prmt(ca[..., 0], cb[..., 0], 0x5410), prmt(ca[..., 0], cb[..., 0], 0x7632),
         prmt(ca[..., 1], cb[..., 1], 0x5410), prmt(ca[..., 1], cb[..., 1], 0x7632)]
    da = ca.view(np.uint16).reshape(100, 32, 4)   # disparities 4l .. 4l + 3 of column a (little-endian halves)
    db = cb.view(np.uint16).reshape(100, 32, 4)
    for k in range(4):
        assert np.array_equal(w[k] & MASK16, da[..., k].astype(np.uint32))
        assert np.array_equal(w[k] >> np.uint32(16), db[..., k].astype(np.uint32))
    assert np.array_equal(prmt(w[0], w[1], 0x5410), ca[..., 0]) and np.array_equal(prmt(w[2], w[3], 0x5410), ca[..., 1])
    assert np.array_equal(prmt(w[0], w[1], 0x7632), cb[..., 0]) and np.array_equal(prmt(w[2], w[3], 0x7632), cb[..., 1])
    # the edge slots carry one column in sgm_step's layout; the mixed input words of the first / last slot
    e = rng.integers(0, 1 << 32, (100, 32, 2), dtype=np.uint64).astype(np.uint32)
    de = e.view(np.uint16).reshape(100, 32, 4)
    a0 = [prmt(e[..., 0], w[0], 0x5410), prmt(e[..., 0], w[1], 0x5432), prmt(e[..., 1], w[2], 0x5410), prmt(e[..., 1], w[3], 0x5432)]
    for k in range(4):   # A of slot 0: (left neighbour's column, low half of the last slot)
        assert np.array_equal(a0[k] & MASK16, de[..., k].astype(np.uint32))
        assert np.array_equal(a0[k] >> np.uint32(16), da[..., k].astype(np.uint32))
    sv = [prmt(w[0], w[1], 0x7632), prmt(w[2], w[3], 0x7632)]   # high half of slot 0, kept before slot 0 moves on
    bl = [prmt(sv[0], e[..., 0], 0x5410), prmt(sv[0], e[..., 0], 0x7632), prmt(sv[1], e[..., 1], 0x5410), prmt(sv[1], e[..., 1], 0x7632)]
    for k in range(4):   # B of the last slot: (high half of slot 0, right neighbour's column)
        assert np.array_equal(bl[k] & MASK16, db[..., k].astype(np.uint32))
        assert np.array_equal(bl[k] >> np.uint32(16), de[..., k].astype(np.uint32))


def vmin_u16x2(*xs):
    lo = np.minimum.reduce([x & MASK16 for x in xs])
    hi = np.minimum.reduce([x >> np.uint32(16) for x in xs])
    return lo | (hi << np.uint32(16))


def vadd2(a, b):
    lo = (a + b) & MASK16
    hi = ((a >> np.uint32(16)) + (b >> np.uint32(16))) & MASK16
    return lo | (hi << np.uint32(16))


def paired_step(I, minI2, Cv, P1, P2):
    """sgm_step_pair restated over a warp: I, Cv [32 lanes][4 words], word k of lane l = disparity 4l + k of recurrence a
    (low half) and b (high half).  __shfl_up_sync(x, 1) hands lane l the value of lane l - 1 (lane 0 keeps its own), so
    that is where the d-1 neighbour of word 0 comes from, and lane 0 -- disparity 0, no d-1 -- takes the all-ones edge
    constant; __shfl_down_sync hands lane l the value of lane l + 1, lane 31 (disparity 127) takes the constant there."""
    u32 = lambda x: (np.asarray(x, np.uint64) & np.uint64(0xffffffff)).astype(np.uint32)
    lane = np.arange(32)
    ones = np.uint64(0xffffffff)
    p1x2 = np.uint64(P1 * 0x10001)
    k2 = np.uint64((0x10000 - P2) * 0x10001)
    Ip = u32(I.astype(np.uint64) + p1x2)
    up_src = np.where(lane == 0, lane, lane - 1)          # shfl up by 1
    dn_src = np.where(lane == 31, lane, lane + 1)         # shfl down by 1
    upm = np.where(lane == 0, 0, 1).astype(np.uint64); upa = np.where(lane == 0, ones, 0).astype(np.uint64)
    dnm = np.where(lane == 31, 0, 1).astype(np.uint64); dna = np.where(lane == 31, ones, 0).astype(np.uint64)
    up = u32(Ip[up_src, 3].astype(np.uint64) * upm + upa)
    dn = u32(Ip[dn_src, 0].astype(np.uint64) * dnm + dna)
    nd2 = u32(np.uint64(minI2) * ones + k2)
    L = np.empty_like(I)
    for k in range(4):
        t = vmin_u16x2(I[:, k], Ip[:, k - 1] if k else up, Ip[:, k + 1] if k < 3 else dn)
        L[:, k] = vmin_u16x2(vadd2(t, vadd2(Cv[:, k], np.full(32, nd2, np.uint32))), Cv[:, k])
    mn = vmin_u16x2(L[:, 0], L[:, 1], L[:, 2], L[:, 3])
    hi = mn.min()
    lo = u32(mn.astype(np.uint64) << np.uint64(16)).min()
    return L, int(prmt(np.array([lo], np.uint32), np.array([hi], np.uint32), 0x7632)[0])


def test_paired_step_equals_the_sgm_recurrence():
    """Several steps of the restated paired step against OpenCV's recurrence on two independent 128-disparity vectors:
    L[d] = C[d] + min(L'[d], L'[d -+ 1] + P1, min L' + P2) - (min L' + P2), no neighbour beyond disparities 0 and 127."""
    P1, P2 = 1944, 7776
    rng = np.random.default_rng(11)
    ref = [np.zeros(128, np.int64), np.zeros(128, np.int64)]
    state = np.zeros((32, 4), np.uint32)
    m2 = 0
    for _ in range(12):
        c = [rng.integers(P2, P2 + 15000, 128), rng.integers(P2, P2 + 15000, 128)]
        c[1][:40] = rng.integers(P2 + 20000, P2 + 24000, 40)   # very different minima in the two halves
        Cv = (c[0].reshape(32, 4) | (c[1].reshape(32, 4) << 16)).astype(np.uint32)
        state, m2 = paired_step(state, m2, Cv, P1, P2)
        for h in range(2):
            prev = ref[h]
            nb = np.full(128, 1 << 40, np.int64)
            nb[1:] = np.minimum(nb[1:], prev[:-1] + P1)
            nb[:-1] = np.minimum(nb[:-1], prev[1:] + P1)
            delta = prev.min() + P2
            ref[h] = c[h] + np.minimum(np.minimum(prev, nb), delta) - delta
        assert np.array_equal((state & MASK16).reshape(-1), ref[0])
        assert np.array_equal((state >> np.uint32(16)).reshape(-1), ref[1])
        assert m2 == int(ref[0].min()) | (int(ref[1].min()) << 16)


# width1 = W - 128 columns -> (CTAs per cluster, columns per warp, last strip full) as sgbm_vwave.cu's vwave_shape picks them
GEOMS = [
    (638, 8, 4, False),     # width1 510
    (828, 8, 6, False),     # width1 700
    (992, 9, 6, True),      # width1 864 = 9 x 16 x 6
    (1129, 8, 8, False),    # width1 1001
    (1280, 9, 8, True),     # width1 1152: config 3's shape
    (1628, 16, 6, True),    # width1 1500
    (729, 8, 5, False),     # width1 601 (odd: the unpaired form)
    (978, 8, 7, False),     # width1 850
    (1228, 8, 9, False),    # width1 1100
]


def scene(W, H, D, seed, kind):
    from laser_3d_reconstruction_b200 import synth
    l, r = synth.stereo_pair(W, H, D, seed)
    if kind == "stripes":
        # columns in stripes of four alternate between the matched scene and anti-correlated noise, so that the two
        # columns sharing a word (p and p + CPW / 2) see very different path minima
        noise = np.random.default_rng(seed).integers(0, 256, (H, W, 3), dtype=np.uint8)
        sel = ((np.arange(W) // 4) % 2 == 1)[None, :, None]
        l = np.where(sel, noise, l).astype(np.uint8)
        r = np.where(sel, 255 - noise, r).astype(np.uint8)
    elif kind == "noise":
        # anti-correlated full-contrast noise at block 11: costs near the top of the int16 domain in every pixel
        noise = np.random.default_rng(seed).integers(0, 256, (H, W, 3), dtype=np.uint8)
        l, r = noise, (255 - noise).astype(np.uint8)
    return np.ascontiguousarray(l), np.ascontiguousarray(r)


def run_pipeline(ctx, W, H, D, bs, frames, lanes, **kw):
    """disp16 of every frame, the maps, and the set of (columns per warp, last strip full) of the wavefront kernels the run
    launched (empty when it ran none), read from the kernel names."""
    import re
    from torch.profiler import ProfilerActivity, profile
    from laser_3d_reconstruction_b200 import _native as N
    from laser_3d_reconstruction_b200 import pipeline, synth
    K, Q = synth.camera_model(W, H)
    maps = synth.warp_maps(W, H, 0) + synth.warp_maps(W, H, 1)
    saved = os.environ.get("L3D_VWAVE")
    os.environ["L3D_VWAVE"] = "1"   # the wavefront kernel wherever it applies (read when a pipeline is created)
    try:
        cfg = pipeline.make_pipeline_config(W, H, D, bs, 1, Q, K, extractor=N.STEGER_IMPROVED, lanes=lanes, max_points=8000, **kw)
        fp = pipeline.FramePipeline(cfg, maps=maps, ctx=ctx)
        try:
            L = np.stack([f[0] for f in frames])
            R = np.stack([f[1] for f in frames])
            dl, dr = fp.upload(L), fp.upload(R)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                fp.run_dev(dl, dr, len(frames))
            shapes = set()
            for e in prof.events():
                m = re.search(r"sgbm_vwave_kernel<(\d+), (\d+), (true|false), (true|false), (\d+)>", e.name)
                if m:
                    assert int(m.group(1)) == D // 64
                    shapes.add((int(m.group(2)), m.group(4) == "true"))
            return [fp.fetch(i)["disp16"] for i in range(len(frames))], maps, shapes
        finally:
            fp.close()
    finally:
        if saved is None:
            os.environ.pop("L3D_VWAVE", None)
        else:
            os.environ["L3D_VWAVE"] = saved


def cv2_disp(frame, maps, params):
    lg = cv2.cvtColor(cv2.remap(frame[0], maps[0], maps[1], cv2.INTER_LINEAR), cv2.COLOR_BGR2GRAY)
    rg = cv2.cvtColor(cv2.remap(frame[1], maps[2], maps[3], cv2.INTER_LINEAR), cv2.COLOR_BGR2GRAY)
    return cv2.StereoSGBM_create(**params).compute(lg, rg)


def check_geometry(ctx, W, H, bs, kind, seed, cpw, full):
    D = 128
    frames = [scene(W, H, D, seed + i, kind) for i in range(9)]
    base, mutated, _ = ref_ops.sgbm_param_sets(D, bs, 1)
    # one matcher, uniquenessRatio 10 (as constructed) and 0 (as the WLS filter leaves it), grouped (15 lanes: one job per
    # frame, so a lane set must have at least 8 frames for the cluster kernels): bit for bit against cv2
    for params, kw in ((base, dict(use_wls=False)), (mutated, dict(use_wls=False, mutated_left=True))):
        got, maps, shapes = run_pipeline(ctx, W, H, D, bs, frames, 15, **kw)
        assert shapes == {(cpw, full)}, "%dx%d: wavefront kernels launched %s, expected %d columns per warp" % (W, H, shapes, cpw)
        for i in (0, 8):
            want = cv2_disp(frames[i], maps, params)
            assert np.array_equal(got[i], want), "%s %dx%d bs %d uniqueness %d frame %d: %d pixels differ from cv2" % (
                kind, W, H, bs, params["uniquenessRatio"], i, int((got[i] != want).sum()))
    # WLS: the left and the right matcher (uniquenessRatio 0) through the wavefront kernel == the lane-per-frame pipeline
    grouped, _, shapes = run_pipeline(ctx, W, H, D, bs, frames, 14)
    assert shapes == {(cpw, full)}, "%dx%d WLS: wavefront kernels launched %s" % (W, H, shapes)
    per_lane, _, shapes = run_pipeline(ctx, W, H, D, bs, frames, 2)
    assert not shapes
    for i in range(len(frames)):
        assert np.array_equal(grouped[i], per_lane[i]), "%s %dx%d WLS frame %d: grouped != lane-per-frame" % (kind, W, H, i)


@pytest.mark.gpu
@pytest.mark.parametrize("W,cluster,cpw,full", GEOMS)
def test_vwave_geometries_bit_exact(ctx, W, cluster, cpw, full):
    assert ((W - 128) % cpw == 0) == full
    check_geometry(ctx, W, 40, 9, "scene", 100 + W, cpw, full)


@pytest.mark.gpu
@pytest.mark.parametrize("W,cpw,full", [(1129, 8, False), (1280, 8, True)])
def test_vwave_paired_columns_with_different_minima(ctx, W, cpw, full):
    check_geometry(ctx, W, 36, 5, "stripes", 300 + W, cpw, full)


@pytest.mark.gpu
@pytest.mark.parametrize("W,cpw,full", [(828, 6, False), (1280, 8, True)])
def test_vwave_paired_costs_near_int16_top(ctx, W, cpw, full):
    check_geometry(ctx, W, 32, 11, "noise", 500 + W, cpw, full)
