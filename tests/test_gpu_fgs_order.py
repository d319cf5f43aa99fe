"""The partitioned parallel FGS solver of the WLS filter (csrc/wls.cu fgsp_solve_line) against its numpy float32
restatement (fgs_f32_partitioned), bit for bit.

The build uses --fmad=false, so every f32 operation of the kernels is executed in source order and rounds once; the
restatement repeats that order.  This pins the solver's operation order: a kernel change that stages, stores or
schedules the solves differently must leave every float of the solution unchanged.
(a) The kernels alone (l3d_fgs_solve) at every chunking regime of test_gpu_fgs.PAR_N, row and column passes, with
    the three lambda schedules.
(b) The whole filter (l3d_wls_filter, parallel solver): its int16 output equals wls_finalize restated in float32 on
    the restated solve of the filter's own confidence map.
(c) On the CPU: the restatement is within test_gpu_fgs's K bounds of the float64 solve."""
import cv2
import numpy as np
import pytest

from laser_3d_reconstruction_b200 import _native as N
from laser_3d_reconstruction_b200 import synth
from oracle import ref_ops
from test_gpu_fgs import K_FLAT, K_PAR, KINDS, LAM, PAR_CASES, SCHEDULES, WLS_SIZES, EPS, line_errors, line_planes


# ---- the restatement ----------------------------------------------------------------------------------------------
def _solve_lines_par_f32(g1, g2, wgt, lam):
    """wls.cu fgsp_solve_line (the partitioned parallel solver) restated in numpy float32, every line of a pass at once:
    g1, g2 (lines, n) right-hand sides, wgt (lines, n) coupling weights.  The line is split into 32 chunks of m =
    max(2, ceil(n / 32)) | 1 elements, one per warp lane; a (lines, 32) array holds one value per lane, and every float32
    operation rounds once, in the kernel's order (__frcp_rn(x) = 1 / x).  -> (g1, g2) solved"""
    f = np.float32
    one, lam = f(1), f(lam)
    L, n = wgt.shape
    m = max(2, -(-n // 32)) | 1
    N = 32 * m
    cnt = np.clip(n - np.arange(32) * m, 0, m)                   # elements of each lane's chunk [s, e]
    act = cnt > 0

    def lanes(x):  # (L, n) -> (L, 32, m), zero past the line's end
        return np.concatenate([x, np.zeros((L, N - n), f)], 1).reshape(L, 32, m)

    c = lam * np.asarray(wgt, f)
    a = np.concatenate([np.zeros((L, 1), f), c[:, :-1]], 1)      # a_j = lam wgt[j - 1], 0 at j = 0
    c, a, r1, r2 = lanes(c), lanes(a), lanes(np.asarray(g1, f)), lanes(np.asarray(g2, f))
    b = (one - a) - c
    with np.errstate(divide="ignore", invalid="ignore", over="ignore", under="ignore"):
        # up sweep: row s as E u_{s-1} + u_s + G u_e = H
        E, G = np.zeros((L, 32), f), np.full((L, 32), -one)
        H1, H2 = np.zeros((L, 32), f), np.zeros((L, 32), f)
        for k in range(m - 2, -1, -1):
            on = k <= cnt - 2
            ck = c[:, :, k]
            ib = one / (b[:, :, k] - ck * E)
            E = np.where(on, a[:, :, k] * ib, E)
            G = np.where(on, ((-ck) * G) * ib, G)
            H1 = np.where(on, (r1[:, :, k] - ck * H1) * ib, H1)
            H2 = np.where(on, (r2[:, :, k] - ck * H2) * ib, H2)
        # down sweep: row j as AB_j u_{s-1} + u_j + D_j u_{j+1} = g_j
        Dd, AB = np.zeros((L, 32, m), f), np.zeros((L, 32, m), f)
        Dp, ABp = np.zeros((L, 32), f), np.full((L, 32), -one)
        p1, p2 = np.zeros((L, 32), f), np.zeros((L, 32), f)
        for k in range(m):
            on = k < cnt
            ak = a[:, :, k]
            ib = one / (b[:, :, k] - ak * Dp)
            Dp = np.where(on, c[:, :, k] * ib, Dp)
            ABp = np.where(on, ((-ak) * ABp) * ib, ABp)
            p1 = np.where(on, (r1[:, :, k] - ak * p1) * ib, p1)
            p2 = np.where(on, (r2[:, :, k] - ak * p2) * ib, p2)
            Dd[:, :, k], AB[:, :, k], r1[:, :, k], r2[:, :, k] = Dp, ABp, p1, p2

        def down(x, d, fill):  # __shfl_down_sync(x, d) with lanes past 31 replaced by `fill`
            return np.concatenate([x[:, d:], np.full((L, d), fill, f)], 1)

        def up(x, d, fill):    # __shfl_up_sync(x, d) with lanes below d replaced by `fill`
            return np.concatenate([np.full((L, d), fill, f), x[:, :-d]], 1)

        # reduced system over the chunk ends: A u_e(l-1) + B u_e(l) + Cc u_e(l+1) = F
        ncnt = np.append(cnt[1:], 0)
        A = np.where(act, ABp, f(0))
        F1, F2 = np.where(act, p1, f(0)), np.where(act, p2, f(0))
        B, Cc = np.ones((L, 32), f), np.zeros((L, 32), f)
        one_next = act & (ncnt == 1)
        more = act & (ncnt > 1)
        Cc = np.where(one_next, Dp, Cc)
        En, Gn, H1n, H2n = down(E, 1, 0), down(G, 1, 0), down(H1, 1, 0), down(H2, 1, 0)
        B = np.where(more, one - Dp * En, B)
        Cc = np.where(more, (-Dp) * Gn, Cc)
        F1 = np.where(more, p1 - Dp * H1n, F1)
        F2 = np.where(more, p2 - Dp * H2n, F2)
        dist = 1
        while dist < 32:  # parallel cyclic reduction
            Am, Bm, Cm, F1m, F2m = up(A, dist, 0), up(B, dist, 1), up(Cc, dist, 0), up(F1, dist, 0), up(F2, dist, 0)
            Ap, Bp, Cp, F1p, F2p = down(A, dist, 0), down(B, dist, 1), down(Cc, dist, 0), down(F1, dist, 0), down(F2, dist, 0)
            k1, k2 = A * (one / Bm), Cc * (one / Bp)
            B = (B - Cm * k1) - Ap * k2
            F1 = (F1 - F1m * k1) - F1p * k2
            F2 = (F2 - F2m * k1) - F2p * k2
            A = (-Am) * k1
            Cc = (-Cp) * k2
            dist <<= 1
        ib = one / B
        ue1, ue2 = F1 * ib, F2 * ib
        up1, up2 = up(ue1, 1, 0), up(ue2, 1, 0)
        # back sweep: u_j = g_j - AB_j u_{s-1} - D_j u_{j+1}
        li = np.arange(32)
        r1[:, li[act], cnt[act] - 1] = ue1[:, act]
        r2[:, li[act], cnt[act] - 1] = ue2[:, act]
        n1, n2 = ue1, ue2
        for k in range(m - 2, -1, -1):
            on = k <= cnt - 2
            n1 = np.where(on, (r1[:, :, k] - AB[:, :, k] * up1) - Dd[:, :, k] * n1, n1)
            n2 = np.where(on, (r2[:, :, k] - AB[:, :, k] * up2) - Dd[:, :, k] * n2, n2)
            r1[:, :, k] = np.where(on, n1, r1[:, :, k])
            r2[:, :, k] = np.where(on, n2, r2[:, :, k])
    return r1.reshape(L, N)[:, :n], r2.reshape(L, N)[:, :n]


def fgs_f32_partitioned(num, den, ch, cv, lam, iters=3, variant=0):
    """The GPU's partitioned parallel FGS solver (wls.cu fgsp_solve_line and dev_fgs's lambda schedule) restated in numpy
    float32, vectorised over lines and lanes: `iters` x (row pass with ch, column pass with cv) on the (h, w) planes num
    and den.  -> (num, den) float32"""
    n1, n2 = np.asarray(num, np.float32), np.asarray(den, np.float32)
    ch, cv = np.asarray(ch, np.float32), np.asarray(cv, np.float32)
    for lh, lv in ref_ops._fgs_lams(lam, iters, variant, np.float32):
        n1, n2 = _solve_lines_par_f32(n1, n2, ch, lh)
        n1, n2 = _solve_lines_par_f32(n1.T, n2.T, cv.T, lv)
        n1, n2 = n1.T, n2.T
    return np.ascontiguousarray(n1), np.ascontiguousarray(n2)


def assert_same(got, want, what):
    bad = np.argwhere(got.view(np.uint32) != want.view(np.uint32))
    assert len(bad) == 0, "%s: %d of %d differ, first at %s: %r vs %r" % (
        what, len(bad), got.size, tuple(bad[0]), got[tuple(bad[0])], want[tuple(bad[0])])


# ---- (a) the kernels alone ----------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("iters,variant", SCHEDULES)
@pytest.mark.parametrize("n,orient", PAR_CASES)
def test_parallel_kernels_bit_identical(ctx, n, orient, iters, variant):
    rng = np.random.default_rng(2000 * n + (orient == "cols") * 7 + iters + 10 * variant)
    num, den, ch, cv = line_planes(rng, n, 3, orient)
    gn, gd, par = ctx.fgs_solve(num, den, ch, cv, LAM, iters, variant)
    assert par, "the partitioned kernels did not run at %s" % (num.shape,)
    wn, wd = fgs_f32_partitioned(num, den, ch, cv, LAM, iters, variant)
    assert_same(gn, wn, "num %s" % (num.shape,))
    assert_same(gd, wd, "den %s" % (num.shape,))


# ---- (b) the whole filter -----------------------------------------------------------------------------------------
def finalize_f32(num, den):
    """wls_finalize_kernel: num * (1 / (den + 1e-43)) in f32 -> int16, half-even, saturated, INT_MIN on NaN / |v| >= 2^31"""
    f = np.float32
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        v = num * (f(1) / (den + f(1e-43)))
        q = np.rint(np.clip(np.nan_to_num(v, nan=0.0), -32768, 32767)).astype(np.int16)
        q[~(np.abs(v) < f(2147483648.0))] = -32768
    return q


def check_filter(ctx, lg, rg, D, bs):
    base, mut, right = ref_ops.sgbm_param_sets(D, bs, 1)
    dl = cv2.StereoSGBM_create(**mut).compute(lg, rg)
    dr = cv2.StereoSGBM_create(**right).compute(rg, lg)
    r = int(np.ceil(0.5 * bs))
    out, conf = ctx.wls_filter(N.WlsParams(LAM, 1.5, 0, D, r, 24, N.WLS_SOLVER_PARALLEL), dl, dr, lg, want_conf=True)
    c = conf[:, D:]
    ch, cv = ref_ops.wls_weights(lg[:, D:], 1.5)
    num, den = fgs_f32_partitioned(c * dl[:, D:].astype(np.float32), c, ch, cv, LAM, 3)
    want = finalize_f32(num, den)
    bad = np.argwhere(out[:, D:] != want)
    assert len(bad) == 0, "%d of %d pixels differ, first at %s" % (len(bad), want.size, tuple(bad[0]))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c1", "c3", "c4"])
def test_wls_filter_bit_identical(ctx, name):
    W, H, D, bs = WLS_SIZES[name]
    l, r = synth.stereo_pair(W, H, D, 9)
    check_filter(ctx, cv2.cvtColor(l, cv2.COLOR_BGR2GRAY), cv2.cvtColor(r, cv2.COLOR_BGR2GRAY), D, bs)


@pytest.mark.gpu
def test_wls_filter_bit_identical_real_pairs(ctx, golden_real):
    for tag in ("a", "b"):
        lg = cv2.cvtColor(golden_real["lrect_" + tag], cv2.COLOR_BGR2GRAY)
        rg = cv2.cvtColor(golden_real["rrect_" + tag], cv2.COLOR_BGR2GRAY)
        check_filter(ctx, lg, rg, 64, 5)


# ---- (c) the restatement against float64 --------------------------------------------------------------------------
@pytest.mark.parametrize("n,orient", [(2, "rows"), (4, "cols"), (94, "rows"), (97, "cols"), (156, "rows"), (1152, "rows")])
def test_restatement_vs_f64(n, orient):
    """The restatement's per-line error against float64 is within the bounds test_gpu_fgs holds the kernels to."""
    rng = np.random.default_rng(3000 * n + (orient == "cols"))
    num, den, ch, cv = line_planes(rng, n, 3, orient)
    wn, wd = ref_ops.fgs_f64(num, den, ch, cv, LAM, 3)
    pn, pd = fgs_f32_partitioned(num, den, ch, cv, LAM, 3)
    sn, sd = ref_ops.fgs_f32_serial(num, den, ch, cv, LAM, 3)
    err_par = np.stack([line_errors(pn, wn, orient), line_errors(pd, wd, orient)]).reshape(2, len(KINDS), -1)
    err_ser = np.stack([line_errors(sn, wn, orient), line_errors(sd, wd, orient)]).reshape(2, len(KINDS), -1)
    k = np.array([K_FLAT if kind == "flat" else K_PAR for kind in KINDS])[None, :, None]
    assert (err_par <= k * err_ser.max(axis=2, keepdims=True) + 8 * EPS).all()
