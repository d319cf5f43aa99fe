// wls.cu -- K3: confidence-weighted WLS disparity filter + K5a disparity -> depth.
// Replaces wls_filter.filter(dl, left_gray, disparity_map_right=dr) and the depth conversion of
// the reference (camera/single_usb_stereo_camera.py:277-282 setup, :328-346).
//
// cv2.ximgproc is absent from the image, so this follows the published opencv_contrib algorithm
// (disparity_filters.cpp + fgs_filter.cpp) as restated in oracle/csrc/orc_wls.c; every f32
// operation is issued unfused and in the oracle's order, so the two agree bit for bit.
//
// Stages (ROI = columns [x0, W), x0 = max(0, minD + numD)):
//   wls_hbox / wls_vbox_conf   (2r+1)^2 box mean of d and d^2 -> variance -> 1 - 0.001 var
//   wls_lrc                    LR-consistency confidence, FGS right-hand sides, guide weights
//   fgs_hpass / fgs_vpass      3 x (row solves, column solves), Thomas algorithm, one line per
//                              thread, numerator and denominator solved together
//   fgs_*_par                  the same solves partitioned over the 32 lanes of a warp (default)
//   wls_finalize               num/(den+eps) -> int16 (half-even, saturated); in the frame pipeline also the depth
#include "common.cuh"

namespace l3d {

__device__ __forceinline__ int reflect101(int p, int n) {
    if (n == 1) return 0;
    while (p < 0 || p >= n) p = p < 0 ? -p : 2 * n - 2 - p;
    return p;
}

// horizontal (2r+1) sums of d and d*d for the left ROI (x0..) and the right ROI (0..)
// full: the taps come from the whole image row (reflected at the image border) instead of the ROI copy (L3D_WLS_BOX_FULL_IMAGE)
__global__ void wls_hbox_kernel(const int16_t* __restrict__ dl, const int16_t* __restrict__ dr, int W, int x0,
                                int w, int h, int r, int full, float* __restrict__ aL, float* __restrict__ bL,
                                float* __restrict__ aR, float* __restrict__ bR) {
    int x = blockIdx.x * blockDim.x + threadIdx.x;
    int y = blockIdx.y;
    if (x >= w) return;
    const int16_t* rl = dl + (size_t)y * W + x0;
    const int16_t* rr = dr + (size_t)y * W;
    float sa = 0.f, sb = 0.f, ta = 0.f, tb = 0.f;
    for (int k = -r; k <= r; k++) {
        float v, u;
        if (full) {
            v = (float)dl[(size_t)y * W + reflect101(x0 + x + k, W)];
            u = (float)dr[(size_t)y * W + reflect101(x + k, W)];
        } else {
            const int xx = reflect101(x + k, w);
            v = (float)rl[xx]; u = (float)rr[xx];
        }
        sa = __fadd_rn(sa, v); sb = __fadd_rn(sb, __fmul_rn(v, v));
        ta = __fadd_rn(ta, u); tb = __fadd_rn(tb, __fmul_rn(u, u));
    }
    size_t i = (size_t)y * w + x;
    aL[i] = sa; bL[i] = sb; aR[i] = ta; bR[i] = tb;
}

__global__ void wls_vbox_conf_kernel(const float* __restrict__ aL, const float* __restrict__ bL,
                                     const float* __restrict__ aR, const float* __restrict__ bR, int w, int h,
                                     int r, int clamp1, float* __restrict__ cl, float* __restrict__ cr) {
    int x = blockIdx.x * blockDim.x + threadIdx.x;
    int y = blockIdx.y;
    if (x >= w) return;
    const float inv = __fdiv_rn(1.0f, (float)((2 * r + 1) * (2 * r + 1)));
    float sa = 0.f, sb = 0.f, ta = 0.f, tb = 0.f;
    for (int k = -r; k <= r; k++) {
        size_t j = (size_t)reflect101(y + k, h) * w + x;
        sa = __fadd_rn(sa, aL[j]); sb = __fadd_rn(sb, bL[j]);
        ta = __fadd_rn(ta, aR[j]); tb = __fadd_rn(tb, bR[j]);
    }
    float ma = __fmul_rn(sa, inv), mb = __fmul_rn(sb, inv);
    float c = __fsub_rn(1.0f, __fmul_rn(0.001f, __fsub_rn(mb, __fmul_rn(ma, ma))));
    size_t i = (size_t)y * w + x;
    if (clamp1 && c > 1.f) c = 1.f;
    cl[i] = c < 0.f ? 0.f : c;
    ma = __fmul_rn(ta, inv); mb = __fmul_rn(tb, inv);
    c = __fsub_rn(1.0f, __fmul_rn(0.001f, __fsub_rn(mb, __fmul_rn(ma, ma))));
    if (clamp1 && c > 1.f) c = 1.f;
    cr[i] = c < 0.f ? 0.f : c;
}

__global__ void wls_lrc_kernel(const int16_t* __restrict__ dl, const int16_t* __restrict__ dr,
                               const uint8_t* __restrict__ guide, const float* __restrict__ lut, int W, int x0,
                               int w, int h, int thresh, int outside_zero, const float* __restrict__ cl, const float* __restrict__ cr,
                               float* __restrict__ conf, float* __restrict__ num, float* __restrict__ den,
                               float* __restrict__ ch, float* __restrict__ cv) {
    int x = blockIdx.x * blockDim.x + threadIdx.x;
    int y = blockIdx.y;
    if (x >= w) return;
    size_t i = (size_t)y * w + x;
    int j = x0 + x;
    int l = dl[(size_t)y * W + j];
    int ridx = j - (l >> 4);
    float c = cl[i];
    if (ridx >= 0 && ridx < w) {
        int rr = dr[(size_t)y * W + ridx];
        if (abs(l + rr) < thresh) c = fminf(c, cr[(size_t)y * w + ridx]);
        else c = 0.f;
    } else if (outside_zero) c = 0.f;
    c = __fmul_rn(255.0f, c);
    conf[i] = c;
    num[i] = __fmul_rn(c, (float)l);
    den[i] = c;
    int g = guide[(size_t)y * W + j];
    float wx = 0.f, wy = 0.f;
    if (x < w - 1) { int d = g - (int)guide[(size_t)y * W + j + 1]; wx = lut[d * d]; }
    if (y < h - 1) { int d = g - (int)guide[(size_t)(y + 1) * W + j]; wy = lut[d * d]; }
    ch[i] = wx; cv[i] = wy;
}

// Thomas solves of one FGS pass (forward elimination + back substitution of every line), identical
// op order to oracle/csrc/orc_wls.c, as THREE lock-step lanes per line:
//   role 0  elimination factors  dn_j = (1 - lam (c_{j-1} + c_j)) - (lam c_{j-1}) D_{j-1},  D_j = (lam c_j) / dn_j
//   role 1  numerator plane      a_j  = (a_j - (lam c_{j-1}) a_{j-1}) / dn_j
//   role 2  denominator plane    the same on den
// Roles 1/2 run one element behind role 0 and receive (dn, lam c_{j-1}) of their element by warp shuffle, so
// a step costs the warp ONE IEEE division sequence for all three quotients and the serial chain per
// element is fmul -> fsub -> fdiv.  The zero initial state reproduces the oracle's special-cased first
// element bit for bit (x + 0, x - 0 and 0 * 0 are exact).  A warp carries LPW lines.  This kernel is the
// vertical pass: lines are image columns, a step reads and writes three runs of LPW adjacent floats
// straight from/to global memory -- no shared memory, one-warp CTAs (116 at config 3), so the solver leaves
// every SM free for the matcher kernels of the other frames in flight.  D goes to a scratch plane for the
// back substitution (role 0 reloads it and shuffles it to roles 1/2).
constexpr int FGS_LPW = 10;   // lines per warp: lanes [0,10) role 0, [10,20) role 1, [20,30) role 2
constexpr int FGS_CPW = 8;    // columns per warp in the vertical pass
constexpr int FGS_BLK = 16;   // elements per register block (the next block is prefetched during the current one)

// LPW: columns per warp (8: each role's run of floats is exactly one aligned 32-byte sector per step)
template <int LPW>
__global__ void __launch_bounds__(32) fgs_cols_kernel(float* num, float* den, const float* __restrict__ wgt,
                                                       float* Dscr, int w, int h, float lam) {
    const int nlines = w, len = h;  // lines are image columns (the row pass is fgs_rows_kernel below)
    const int lane = threadIdx.x;
    const int role = lane / LPW, li = lane - role * LPW;
    const int line = min(blockIdx.x * LPW + li, nlines - 1);
    const bool active = role < 3 && blockIdx.x * LPW + li < nlines;
    const int src = li;                                   // role-0 lane of this lane's line
    const size_t ls = 1, es = (size_t)w;
    const float* in = role == 0 ? wgt : (role == 1 ? num : den);
    float* out = role == 0 ? Dscr : (role == 1 ? num : den);
    in += (size_t)line * ls; out += (size_t)line * ls;
    const int lag = role == 0 ? 0 : 1;
    const bool r0 = role == 0;
    // ---- forward elimination: steps j = 0 .. len (roles 1/2 finish element len-1 in step len)
    float p = 0.f, cm = 0.f;              // previous quotient (D or a), previous weight (role 0)
    float dn_pub = 1.f, lcm_pub = 0.f;    // role 0: dn and lam*c_{j-1} of the element it processed last
    float xs[FGS_BLK], xn[FGS_BLK];
    auto load_blk = [&](float (&dst)[FGS_BLK], int j0) {
#pragma unroll
        for (int k = 0; k < FGS_BLK; k++) {
            const int e = j0 + k - lag;
            dst[k] = (e >= 0 && e < len) ? in[(size_t)e * es] : 0.f;
        }
    };
    load_blk(xs, 0);
    for (int j0 = 0; j0 <= len; j0 += FGS_BLK) {
        if (j0 + FGS_BLK <= len) load_blk(xn, j0 + FGS_BLK);
#pragma unroll
        for (int k = 0; k < FGS_BLK; k++) {
            const int e = j0 + k - lag;
            const float x = xs[k];
            const float dn_s = __shfl_sync(0xffffffffu, dn_pub, src);
            const float lcm_s = __shfl_sync(0xffffffffu, lcm_pub, src);
            const float t = r0 ? __fmul_rn(lam, cm) : lcm_s;
            const float prod = __fmul_rn(t, p);
            const float dn0 = __fsub_rn(__fsub_rn(1.0f, __fmul_rn(lam, __fadd_rn(cm, x))), prod);
            const float numer = r0 ? __fmul_rn(lam, x) : __fsub_rn(x, prod);
            const float denom = r0 ? dn0 : dn_s;
            p = __fdiv_rn(numer, denom);
            if (active && e >= 0 && e < len) out[(size_t)e * es] = p;
            dn_pub = denom; lcm_pub = t; cm = x;
        }
#pragma unroll
        for (int k = 0; k < FGS_BLK; k++) xs[k] = xn[k];
    }
    // ---- back substitution: r_j = r_j - D_j r_{j+1}, j = len-2 .. 0 (p holds r_{len-1} for roles 1/2)
    // roles 1/2 processed element len-1 in the step with e == len-1; later steps of the last block ran on
    // zero inputs with stale (dn, lcm): restore p from memory instead of tracking it through the tail
    if (len >= 1) p = out[(size_t)(len - 1) * es];
    auto load_rev = [&](float (&dst)[FGS_BLK], int j0) {  // elements j0, j0-1, ...
#pragma unroll
        for (int k = 0; k < FGS_BLK; k++) {
            const int e = j0 - k;
            dst[k] = e >= 0 ? out[(size_t)e * es] : 0.f;
        }
    };
    load_rev(xs, len - 2);
    for (int j0 = len - 2; j0 >= 0; j0 -= FGS_BLK) {
        if (j0 - FGS_BLK >= 0) load_rev(xn, j0 - FGS_BLK);
#pragma unroll
        for (int k = 0; k < FGS_BLK; k++) {
            const int e = j0 - k;
            const float Dj = __shfl_sync(0xffffffffu, xs[k], src);
            const float r = __fsub_rn(xs[k], __fmul_rn(Dj, p));
            if (e >= 0 && !r0) {
                p = r;
                if (active) out[(size_t)e * es] = r;
            }
        }
#pragma unroll
        for (int k = 0; k < FGS_BLK; k++) xs[k] = xn[k];
    }
}

// Horizontal pass of the same solver.  Ten rows per warp would read and write 4 scattered bytes per lane
// and step (one 32-byte sector per useful float, every step of every frame in flight -- measured: a tenth of
// the whole pipeline's throughput), so the rows move through shared memory in 32-column tiles: 30 coalesced
// 128-byte cp.async requests bring the next tile of the 3 x 10 row segments in while the current one is being
// eliminated, results overwrite their inputs in the ring and leave as coalesced 128-byte stores one tile later.
constexpr int FGS_T = 32;               // tile columns
constexpr int FGS_RING = 3 * FGS_T;     // ring of three tiles per row segment (processing / prefetch / draining)
constexpr int FGS_RS = FGS_RING + 1;    // padded segment stride: the 30 lanes of a step hit 30 different banks
constexpr int FGS_NSEG = 3 * FGS_LPW;

__global__ void __launch_bounds__(32) fgs_rows_kernel(float* num, float* den, const float* __restrict__ wgt,
                                                      float* Dscr, int w, int h, float lam) {
    __shared__ float ring[FGS_NSEG * FGS_RS];
    const int lane = threadIdx.x;
    const int role = lane / FGS_LPW, li = lane - role * FGS_LPW;
    const int row0 = blockIdx.x * FGS_LPW;
    const int nrows = min(FGS_LPW, h - row0);
    const bool active = role < 3 && li < nrows;
    const bool r0 = role == 0;
    const int lag = r0 ? 0 : 1;
    const int src = li;
    const int seg = min(role, 2) * FGS_LPW + li;  // lanes 30/31 shadow a real segment (reads only)
    float* const myring = ring + seg * FGS_RS;
    const uint32_t ring_s = (uint32_t)__cvta_generic_to_shared(ring);
    const int ntiles = (w + FGS_T - 1) / FGS_T;
    auto seg_ptr = [&](int i, bool out) -> float* {  // row segment i = plane i / 10, row i % 10 (clamped: duplicates are never stored)
        const int pr = i / FGS_LPW, r = row0 + min(i - pr * FGS_LPW, nrows - 1);
        float* base = pr == 0 ? (out ? Dscr : const_cast<float*>(wgt)) : (pr == 1 ? num : den);
        return base + (size_t)r * w;
    };
    auto load_tile = [&](int T, bool fwd) {  // fwd: weights + num + den; backward: D + num + den
        const int col = T * FGS_T + lane;
        if (col < w) {
#pragma unroll
            for (int i = 0; i < FGS_NSEG; i++) {
                const float* g = seg_ptr(i, !fwd) + col;
                const uint32_t d = ring_s + (uint32_t)(i * FGS_RS + (T % 3) * FGS_T + lane) * 4u;
                asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(g) : "memory");
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto flush_tile = [&](int T, int first_plane) {
        const int col = T * FGS_T + lane;
        if (col < w) {
#pragma unroll
            for (int i = 0; i < FGS_NSEG; i++) {
                if (i < first_plane * FGS_LPW || i - (i / FGS_LPW) * FGS_LPW >= nrows) continue;
                seg_ptr(i, true)[col] = ring[i * FGS_RS + (T % 3) * FGS_T + lane];
            }
        }
    };
    // ---- forward elimination: steps j = 0 .. w, roles 1/2 one element behind role 0 (see fgs_cols_kernel)
    float p = 0.f, cm = 0.f, dn_pub = 1.f, lcm_pub = 0.f;
    const int nsteps_t = (w + 1 + FGS_T - 1) / FGS_T;
    load_tile(0, true);
    for (int T = 0; T < nsteps_t; T++) {
        if (T + 1 < ntiles) {
            load_tile(T + 1, true);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncwarp();
#pragma unroll 8
        for (int k = 0; k < FGS_T; k++) {
            const int e = T * FGS_T + k - lag;
            const bool ok = e >= 0 && e < w;
            const int slot = ok ? e % FGS_RING : 0;
            const float x = ok ? myring[slot] : 0.f;
            const float dn_s = __shfl_sync(0xffffffffu, dn_pub, src);
            const float lcm_s = __shfl_sync(0xffffffffu, lcm_pub, src);
            const float t = r0 ? __fmul_rn(lam, cm) : lcm_s;
            const float prod = __fmul_rn(t, p);
            const float dn0 = __fsub_rn(__fsub_rn(1.0f, __fmul_rn(lam, __fadd_rn(cm, x))), prod);
            const float numer = r0 ? __fmul_rn(lam, x) : __fsub_rn(x, prod);
            const float denom = r0 ? dn0 : dn_s;
            p = __fdiv_rn(numer, denom);
            if (active && ok) myring[slot] = p;
            dn_pub = denom; lcm_pub = t; cm = x;
        }
        __syncwarp();
        if (T >= 1) flush_tile(T - 1, 0);
        __syncwarp();  // the drained slot is the next iteration's prefetch target
    }
    for (int T = nsteps_t - 1; T < ntiles; T++) flush_tile(T, 0);
    __syncwarp();
    // ---- back substitution: r_e = r_e - D_e r_{e+1}, e = w-2 .. 0; role 0 lanes supply D by shuffle
    if (w >= 1) p = myring[(w - 1) % FGS_RING];
    __syncwarp();
    load_tile(ntiles - 1, false);
    for (int T = ntiles - 1; T >= 0; T--) {
        if (T >= 1) {
            load_tile(T - 1, false);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncwarp();
#pragma unroll 8
        for (int k = FGS_T - 1; k >= 0; k--) {
            const int e = T * FGS_T + k;
            const bool ok = e <= w - 2;
            const int slot = e % FGS_RING;
            const float x = ok ? myring[slot] : 0.f;
            const float Dj = __shfl_sync(0xffffffffu, x, src);
            const float r = __fsub_rn(x, __fmul_rn(Dj, p));
            if (ok && !r0) {
                p = r;
                if (active) myring[slot] = r;
            }
        }
        __syncwarp();
        flush_tile(T, 1);
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------
// The same solves as a PARALLEL (partitioned) tridiagonal solver: one warp per line, the line split into 32 chunks.
// The serial kernels above repeat the oracle's operation order (bit-identical, 2 x len dependent division steps
// per line: 1.3 ms per frame at 1280x720, all of it latency); this form has about 3 x len / 32 dependent steps and
// takes the solver off the single-frame critical path.  Results differ from the serial order in the last bits of
// the f32 solution (tolerance class: the int16 output differs by at most 1 LSB, on well under 0.1 % of the pixels).
//
// Line system (fgs_filter.cpp):  a_j u_{j-1} + b_j u_j + c_j u_{j+1} = f_j,  c_j = lam w_j (w = LUT weight <= 0),
// a_j = c_{j-1},  b_j = 1 - a_j - c_j;  two right-hand sides (numerator and denominator plane) share the matrix.
// Lane l owns the chunk [s, e].
//   up sweep    (e-1 .. s, nothing stored): row s as   E u_{s-1} + u_s + G u_e = H
//   down sweep  (s .. e, stored per element): D_j = c_j / beta_j, AB_j = alpha_j / beta_j, g_j = phi_j / beta_j  with
//               beta_j = b_j - a_j D_{j-1}: row j as   AB_j u_{s-1} + u_j + D_j u_{j+1} = g_j
//   reduced system in the chunk ends u_e (one row per lane: row e with u_{s'} of the next chunk replaced by that
//               chunk's row-s form), solved across the lanes by parallel cyclic reduction with warp shuffles
//   back sweep  (e-1 .. s): u_j = g_j - AB_j u_{s-1} - D_j u_{j+1}
// A line lives in shared memory as four planes: weights (overwritten by D in the down sweep), g1, g2 and AB; a lane
// walks its chunk with an odd element stride between lanes, so every step of a sweep hits 32 different banks.  The
// kernels stage their lines with asynchronous copies issued all at once (one bulk copy per row plane, or one cp.async
// per element) instead of a loop of dependent loads: the solves do little arithmetic, and what they cost the frame
// pipeline is the SMs they hold (an SM that hosts an FGS CTA is closed to the matcher kernels, which each need a whole
// register file) times how long they hold them.
constexpr int FGSP_ROWS = 4;        // lines (= warps) per CTA in the row pass
constexpr int FGSP_W_MAX = 2552;    // longest row / column the parallel kernels solve; longer lines take the serial kernels
constexpr int FGSP_H_MAX = 1248;

__device__ __forceinline__ void fgsp_solve_line(float* wd, float* g1, float* g2, float* AB, int n, float lam, int lane) {
    int m = (n + 31) / 32;
    if (m < 2) m = 2;
    m |= 1;                                            // odd chunk length: lane stride == m mod 32 is odd
    const int s = lane * m, e = min(s + m, n) - 1;     // chunk [s, e]; empty when s >= n
    const bool act = s < n;
    const int cnt = act ? e - s + 1 : 0;
    // ---- up sweep: row s in terms of (u_{s-1}, u_s, u_e)
    float E = 0.f, G = -1.f, H1 = 0.f, H2 = 0.f;
    for (int j = e - 1; j >= s && act; j--) {
        const float c = __fmul_rn(lam, wd[j]), a = j > 0 ? __fmul_rn(lam, wd[j - 1]) : 0.f;
        const float b = 1.0f - a - c;
        const float ib = __frcp_rn(b - c * E);
        E = a * ib;
        G = -c * G * ib;
        H1 = (g1[j] - c * H1) * ib;
        H2 = (g2[j] - c * H2) * ib;
    }
    // ---- down sweep: D_j replaces w_j; a_j = lam w_{j-1} is carried from the previous step.  The first a is the
    // previous chunk's last weight, which its lane overwrites: read it before any lane writes D.
    float a = act && s > 0 ? __fmul_rn(lam, wd[s - 1]) : 0.f;
    __syncwarp();
    float Dp = 0.f, ABp = -1.f, p1 = 0.f, p2 = 0.f;
    for (int j = s; j <= e && act; j++) {
        const float c = __fmul_rn(lam, wd[j]);
        const float b = 1.0f - a - c;
        const float ib = __frcp_rn(b - a * Dp);
        Dp = c * ib;
        ABp = -a * ABp * ib;
        p1 = (g1[j] - a * p1) * ib;
        p2 = (g2[j] - a * p2) * ib;
        wd[j] = Dp; AB[j] = ABp; g1[j] = p1; g2[j] = p2;
        a = c;
    }
    // ---- reduced system over the chunk ends: A u_e(l-1) + B u_e(l) + C u_e(l+1) = F
    const int ncnt = __shfl_down_sync(0xffffffffu, cnt, 1);
    const float En = __shfl_down_sync(0xffffffffu, E, 1), Gn = __shfl_down_sync(0xffffffffu, G, 1);
    const float H1n = __shfl_down_sync(0xffffffffu, H1, 1), H2n = __shfl_down_sync(0xffffffffu, H2, 1);
    float A = 0.f, B = 1.f, Cc = 0.f, F1 = 0.f, F2 = 0.f;
    if (act) {
        A = ABp; F1 = p1; F2 = p2;
        const bool has_next = lane < 31 && ncnt > 0;
        if (has_next && ncnt == 1) Cc = Dp;                       // the next chunk's first element is its end
        else if (has_next) { B = 1.0f - Dp * En; Cc = -Dp * Gn; F1 = p1 - Dp * H1n; F2 = p2 - Dp * H2n; }
    }
#pragma unroll
    for (int dist = 1; dist < 32; dist <<= 1) {
        float Am = __shfl_up_sync(0xffffffffu, A, dist), Bm = __shfl_up_sync(0xffffffffu, B, dist);
        float Cm = __shfl_up_sync(0xffffffffu, Cc, dist), F1m = __shfl_up_sync(0xffffffffu, F1, dist), F2m = __shfl_up_sync(0xffffffffu, F2, dist);
        float Ap = __shfl_down_sync(0xffffffffu, A, dist), Bp = __shfl_down_sync(0xffffffffu, B, dist);
        float Cp = __shfl_down_sync(0xffffffffu, Cc, dist), F1p = __shfl_down_sync(0xffffffffu, F1, dist), F2p = __shfl_down_sync(0xffffffffu, F2, dist);
        if (lane < dist) { Am = 0.f; Bm = 1.f; Cm = 0.f; F1m = 0.f; F2m = 0.f; }
        if (lane + dist > 31) { Ap = 0.f; Bp = 1.f; Cp = 0.f; F1p = 0.f; F2p = 0.f; }
        const float k1 = A * __frcp_rn(Bm), k2 = Cc * __frcp_rn(Bp);
        B = B - Cm * k1 - Ap * k2;
        F1 = F1 - F1m * k1 - F1p * k2;
        F2 = F2 - F2m * k1 - F2p * k2;
        A = -Am * k1;
        Cc = -Cp * k2;
    }
    const float ib = __frcp_rn(B);
    const float ue1 = F1 * ib, ue2 = F2 * ib;
    float up1 = __shfl_up_sync(0xffffffffu, ue1, 1), up2 = __shfl_up_sync(0xffffffffu, ue2, 1);
    if (lane == 0) { up1 = 0.f; up2 = 0.f; }
    // ---- back sweep
    if (act) {
        float n1 = ue1, n2 = ue2;
        g1[e] = n1; g2[e] = n2;
        for (int j = e - 1; j >= s; j--) {
            const float d = wd[j], ab = AB[j];
            n1 = g1[j] - ab * up1 - d * n1;
            n2 = g2[j] - ab * up2 - d * n2;
            g1[j] = n1; g2[j] = n2;
        }
    }
}

__device__ __forceinline__ void cp_async4(float* dst, const float* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}

// row plane pitch (floats): a multiple of 4 when w is, so that every plane of a line starts 16-byte aligned
__host__ __device__ inline int fgsp_row_pitch(int w) { return w + 8; }
static size_t fgsp_rows_smem(int w) { return (size_t)FGSP_ROWS * 4 * fgsp_row_pitch(w) * sizeof(float); }

// row pass: warp <-> image row; num / den are solved in place.  bulk (w % 4 == 0 and 16-byte aligned planes): each
// plane row moves as one cp.async.bulk (in on an mbarrier, out as a bulk store); otherwise one cp.async per element.
__global__ void __launch_bounds__(FGSP_ROWS * 32) fgs_rows_par_kernel(float* num, float* den, const float* __restrict__ wgt,
                                                                     int w, int h, float lam, int bulk) {
    extern __shared__ __align__(16) float fsm[];
    __shared__ __align__(8) uint64_t bar[FGSP_ROWS];
    const int LP = fgsp_row_pitch(w);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * FGSP_ROWS + warp;
    if (row >= h) return;  // whole warps; the CTA never synchronises
    float* base = fsm + (size_t)warp * 4 * LP;
    float *sw = base, *s1 = base + LP, *s2 = base + 2 * LP, *sA = base + 3 * LP;
    const size_t off = (size_t)row * w;
    const uint32_t bytes = (uint32_t)w * 4u;
    if (bulk) {
        const uint32_t mb = (uint32_t)__cvta_generic_to_shared(&bar[warp]);
        if (lane == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mb) : "memory");
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(3u * bytes) : "memory");
            const float* src[3] = {wgt + off, num + off, den + off};
            float* dst[3] = {sw, s1, s2};
#pragma unroll
            for (int i = 0; i < 3; i++)
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"((uint32_t)__cvta_generic_to_shared(dst[i])), "l"(src[i]), "r"(bytes), "r"(mb) : "memory");
        }
        __syncwarp();
        asm volatile("{\n\t.reg .pred P1;\n\tWAIT:\n\t"
                     "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], 0;\n\t"
                     "@!P1 bra WAIT;\n\t}" ::"r"(mb) : "memory");
    } else {
        for (int i = lane; i < w; i += 32) {
            cp_async4(sw + i, wgt + off + i); cp_async4(s1 + i, num + off + i); cp_async4(s2 + i, den + off + i);
        }
        asm volatile("cp.async.wait_all;" ::: "memory");
        __syncwarp();
    }
    fgsp_solve_line(sw, s1, s2, sA, w, lam, lane);
    if (bulk) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the solve's stores, visible to the bulk copy
        __syncwarp();
        if (lane == 0) {
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                         ::"l"(num + off), "r"((uint32_t)__cvta_generic_to_shared(s1)), "r"(bytes) : "memory");
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                         ::"l"(den + off), "r"((uint32_t)__cvta_generic_to_shared(s2)), "r"(bytes) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // shared memory stays alive until read
        }
    } else {
        __syncwarp();
        for (int i = lane; i < w; i += 32) { num[off + i] = s1[i]; den[off + i] = s2[i]; }
    }
}

// column plane pitch (floats): == 32 / NC mod 32, so that a staging request (NC adjacent columns x 32 / NC rows) hits
// 32 different banks.  Plane p of column c starts at (p * NC + c) * pitch.
__host__ __device__ inline int fgsp_col_pitch(int h, int nc) { return ((h + 31) / 32) * 32 + 32 / nc; }
static size_t fgsp_cols_smem(int h, int nc) { return (size_t)nc * 4 * fgsp_col_pitch(h, nc) * sizeof(float); }

// column pass: a CTA stages NC adjacent columns (4 NC contiguous bytes per image row), warp <-> column.  The staging
// copies are one cp.async per element, all issued before the one wait: a 16-byte copy would span four columns, which
// live in different planes.
template <int NC>
__global__ void __launch_bounds__(NC * 32) fgs_cols_par_kernel(float* num, float* den, const float* __restrict__ wgt,
                                                              int w, int h, float lam) {
    extern __shared__ __align__(16) float fsm[];
    const int LP = fgsp_col_pitch(h, NC);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int col0 = blockIdx.x * NC;
    const int ncol = min(NC, w - col0);
    const int tc = threadIdx.x % NC, tr = threadIdx.x / NC;  // staging role: column, row phase (32 phases)
    if (tc < ncol) {
        for (int r = tr; r < h; r += 32) {
            const size_t g = (size_t)r * w + col0 + tc;
            cp_async4(fsm + (size_t)tc * LP + r, wgt + g);
            cp_async4(fsm + (size_t)(NC + tc) * LP + r, num + g);
            cp_async4(fsm + (size_t)(2 * NC + tc) * LP + r, den + g);
        }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();
    if (warp < ncol)
        fgsp_solve_line(fsm + (size_t)warp * LP, fsm + (size_t)(NC + warp) * LP, fsm + (size_t)(2 * NC + warp) * LP,
                        fsm + (size_t)(3 * NC + warp) * LP, h, lam, lane);
    __syncthreads();
    if (tc < ncol) {
        const float *s1 = fsm + (size_t)(NC + tc) * LP, *s2 = fsm + (size_t)(2 * NC + tc) * LP;
        for (int r = tr; r < h; r += 32) {
            const size_t g = (size_t)r * w + col0 + tc;
            num[g] = s1[r]; den[g] = s2[r];
        }
    }
}

// ---- K5a: disparity -> depth of one pixel (camera/single_usb_stereo_camera.py:335-357) ------------------------------
struct QMat { double q[16]; };

__device__ __forceinline__ float depth_q_px(int16_t d16, int x, int y, const QMat& Q) {
    float disp = __fdiv_rn((float)d16, 16.0f);
    double d = (double)disp, fx = (double)x, fy = (double)y;
    // cv2.reprojectImageTo3D (4.13, probed): [X Y Z W]^T = Q [x y d 1]^T in f64, the numerator is
    // first stored as f32 (Vec3f), then divided by the f64 W and rounded to f32 again
    double Z = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(Q.q[8], fx), __dmul_rn(Q.q[9], fy)), __dmul_rn(Q.q[10], d)), Q.q[11]);
    double Wh = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(Q.q[12], fx), __dmul_rn(Q.q[13], fy)), __dmul_rn(Q.q[14], d)), Q.q[15]);
    float z = (float)__ddiv_rn((double)(float)Z, Wh);
    if (z < 0.f) z = 0.f;
    if (z > 10.f) z = 0.f;
    if (disp <= 0.f) z = 0.f;
    return z;
}

__device__ __forceinline__ float depth_default_px(int16_t d16) {
    float disp = __fdiv_rn((float)d16, 16.0f);
    float z = 0.f;
    if (disp > 0.f) z = __fdiv_rn((float)(0.06 * 350), disp);
    if (z > 10.f) z = 0.f;
    return z;
}

// DEPTH: 0 = the filtered disparity alone; 1 / 2 = also its depth, through Q / the default baseline (dev_depth's two
// kernels), so the frame pipeline spends no launch and no re-read of the disparity on it
template <int DEPTH>
__global__ void wls_finalize_kernel(const float* __restrict__ num, const float* __restrict__ den,
                                    const float* __restrict__ conf, int W, int H, int x0, int w, int outside,
                                    int16_t* __restrict__ out, float* __restrict__ conf_out, QMat Q, float* __restrict__ depth) {
    int x = blockIdx.x * blockDim.x + threadIdx.x;
    int y = blockIdx.y;
    if (x >= W) return;
    size_t o = (size_t)y * W + x;
    int q;
    if (x < x0) {
        q = outside;
        if (conf_out) conf_out[o] = 0.f;
    } else {
        size_t i = (size_t)y * w + (x - x0);
        float v = __fmul_rn(num[i], __fdiv_rn(1.0f, __fadd_rn(den[i], 1e-43f)));
        if (!(fabsf(v) < 2147483648.f)) q = -32768;  // NaN / |v| >= 2^31: cvRound gives INT_MIN
        else if (v >= 32767.f) q = 32767;
        else if (v <= -32768.f) q = -32768;
        else q = __float2int_rn(v);
        if (conf_out) conf_out[o] = conf[i];
    }
    out[o] = (int16_t)q;
    if (DEPTH == 1) depth[o] = depth_q_px((int16_t)q, x, y, Q);
    if (DEPTH == 2) depth[o] = depth_default_px((int16_t)q);
}

static int wls_finalize(Lane& L, const float* num, const float* den, const float* conf, int W, int H, int x0, int w,
                        int outside, int16_t* out, float* conf_out, float* depth, const double* Q) {
    const dim3 g(cdiv(W, 128), H);
    QMat q{};
    if (Q) memcpy(q.q, Q, sizeof(q.q));
    if (!depth) L3D_LAUNCH(L, wls_finalize_kernel<0>, g, 128, 0, num, den, conf, W, H, x0, w, outside, out, conf_out, q, depth);
    else if (Q) L3D_LAUNCH(L, wls_finalize_kernel<1>, g, 128, 0, num, den, conf, W, H, x0, w, outside, out, conf_out, q, depth);
    else L3D_LAUNCH(L, wls_finalize_kernel<2>, g, 128, 0, num, den, conf, W, H, x0, w, outside, out, conf_out, q, depth);
    return L3D_OK;
}

// exp LUT for the guide weights: lut[k] = -exp(-sqrt(k)/sigma), k = squared grey difference
static int wls_lut(Lane& L, double sigma, float** out) {
    float* dev = L.get<float>(S_WLS_K, 65536);
    if (L.wls_lut_sigma != sigma) {  // per-lane device copy, rebuilt only when sigma changes
        std::vector<float> host(65536);
        for (int i = 0; i < 65536; i++) host[i] = (float)(-exp(-sqrt((double)(float)i) / sigma));
        L3D_CHECK(L, cudaMemcpyAsync(dev, host.data(), 65536 * sizeof(float), cudaMemcpyHostToDevice, L.stream));
        L3D_CHECK(L, cudaStreamSynchronize(L.stream));
        L.wls_lut_sigma = sigma;
    }
    *out = dev;
    return L3D_OK;
}

// The FGS passes of the WLS filter (dev_wls; l3d_fgs_solve runs them alone): `iters` iterations of (row solves with
// weights ch, column solves with weights cv) on num/den in place; Dscr (w x h) is scratch of the serial kernels.
// solver: 0 = partitioned parallel solves (default), 1 = serial solves in the oracle's operation order (bit-identical
// to oracle/csrc/orc_wls.c); L3D_FGS_SERIAL=1 forces the serial form everywhere, and so do lines longer than
// FGSP_W_MAX / FGSP_H_MAX or shorter than 2.
int dev_fgs(Lane& L, int solver, int variant, double lambda, int iters, const float* ch, const float* cv, int w, int h,
            float* num, float* den, float* Dscr, bool* parallel_used) {
    float lam = (float)lambda;
    static const bool force_serial = getenv("L3D_FGS_SERIAL") && atoi(getenv("L3D_FGS_SERIAL")) > 0;
    const bool parallel = !force_serial && solver != 1 && w <= FGSP_W_MAX && h <= FGSP_H_MAX && w >= 2 && h >= 2;
    *parallel_used = parallel;
    const size_t smr = fgsp_rows_smem(w);
    int nc = 8;  // columns per CTA: 16 where a 16-column CTA fits an SM, else 8
    const int bulk = w % 4 == 0 && ((uintptr_t)num | (uintptr_t)den | (uintptr_t)ch) % 16 == 0;
    if (parallel) {
        int dev = 0, optin = 0, fit = 0;
        L3D_CHECK(L, cudaGetDevice(&dev));
        L3D_CHECK(L, cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
        if (fgsp_cols_smem(h, 16) <= (size_t)optin) {
            L3D_CHECK(L, cudaFuncSetAttribute(fgs_cols_par_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fgsp_cols_smem(h, 16)));
            L3D_CHECK(L, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fit, fgs_cols_par_kernel<16>, 16 * 32, fgsp_cols_smem(h, 16)));
        }
        if (fit >= 1) nc = 16;
        else L3D_CHECK(L, cudaFuncSetAttribute(fgs_cols_par_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fgsp_cols_smem(h, 8)));
        L3D_CHECK(L, cudaFuncSetAttribute(fgs_rows_par_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smr));
    }
    const size_t smc = fgsp_cols_smem(h, nc);
    for (int it = 0; it < iters; it++) {
        if (parallel) L3D_LAUNCH(L, fgs_rows_par_kernel, cdiv(h, FGSP_ROWS), FGSP_ROWS * 32, smr, num, den, ch, w, h, lam, bulk);
        else L3D_LAUNCH(L, fgs_rows_kernel, cdiv(h, FGS_LPW), 32, 0, num, den, ch, Dscr, w, h, lam);
        if (variant & L3D_WLS_LAMBDA_PER_PASS) lam *= 0.25f;
        if (parallel && nc == 16) L3D_LAUNCH(L, fgs_cols_par_kernel<16>, cdiv(w, 16), 16 * 32, smc, num, den, cv, w, h, lam);
        else if (parallel) L3D_LAUNCH(L, fgs_cols_par_kernel<8>, cdiv(w, 8), 8 * 32, smc, num, den, cv, w, h, lam);
        else L3D_LAUNCH(L, fgs_cols_kernel<FGS_CPW>, cdiv(w, FGS_CPW), 32, 0, num, den, cv, Dscr, w, h, lam);
        lam *= 0.25f;
    }
    return L3D_OK;
}

int dev_wls(Lane& L, const l3d_wls_params& p, const int16_t* dl, const int16_t* dr, const uint8_t* guide,
            int W, int H, int16_t* out, float* conf_out, float* depth, const double* Q) {
    int x0 = std::max(0, p.min_disp + p.num_disp);
    int w = W - x0, h = H;
    int outside = 16 * (p.min_disp - 1);
    if (w <= 0) {
        // nothing inside the ROI: constant output
        return wls_finalize(L, nullptr, nullptr, nullptr, W, H, W, 0, outside, out, conf_out, depth, Q);
    }
    L3D_ARG(L, p.dd_radius >= 0 && p.dd_radius < 64, "wls dd_radius");
    size_t n = (size_t)w * h;
    float *aL = L.get<float>(S_WLS_A, n), *bL = L.get<float>(S_WLS_B, n), *aR = L.get<float>(S_WLS_C, n), *bR = L.get<float>(S_WLS_D, n);
    float *cl = L.get<float>(S_WLS_E, n), *cr = L.get<float>(S_WLS_F, n);
    float *conf = L.get<float>(S_WLS_G, n), *ch = L.get<float>(S_WLS_H, n), *cv = L.get<float>(S_WLS_I, n);
    float* lut = nullptr;
    int rc = wls_lut(L, p.sigma_color, &lut);
    if (rc != L3D_OK) return rc;
    dim3 g(cdiv(w, 128), h);
    L.t_begin("wls");
    L3D_LAUNCH(L, wls_hbox_kernel, g, 128, 0, dl, dr, W, x0, w, h, p.dd_radius, (p.variant & L3D_WLS_BOX_FULL_IMAGE) ? 1 : 0, aL, bL, aR, bR);
    L3D_LAUNCH(L, wls_vbox_conf_kernel, g, 128, 0, aL, bL, aR, bR, w, h, p.dd_radius, (p.variant & L3D_WLS_CONF_CLAMP_1) ? 1 : 0, cl, cr);
    // aL/bL are free now: reuse as num/den
    float *num = aL, *den = bL;
    L3D_LAUNCH(L, wls_lrc_kernel, g, 128, 0, dl, dr, guide, lut, W, x0, w, h, p.lrc_thresh, (p.variant & L3D_WLS_LRC_OUTSIDE_ZERO) ? 1 : 0, cl, cr, conf, num, den, ch,
               cv);
    bool parallel = false;
    rc = dev_fgs(L, p.solver, p.variant, p.lambda, 3, ch, cv, w, h, num, den, aR, &parallel);  // aR is free as well: scratch D
    if (rc != L3D_OK) return rc;
    rc = wls_finalize(L, num, den, conf, W, H, x0, w, outside, out, conf_out, depth, Q);
    L.t_end("wls");
    if (rc != L3D_OK) return rc;
    return L3D_OK;
}

// ---- K5a: disparity -> depth ---------------------------------------------------------------
__global__ void depth_q_kernel(const int16_t* __restrict__ d16, int W, int H, QMat Q, float* __restrict__ depth) {
    int x = blockIdx.x * blockDim.x + threadIdx.x;
    int y = blockIdx.y;
    if (x >= W) return;
    size_t i = (size_t)y * W + x;
    depth[i] = depth_q_px(d16[i], x, y, Q);
}

__global__ void depth_default_kernel(const int16_t* __restrict__ d16, size_t n, float* __restrict__ depth) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    depth[i] = depth_default_px(d16[i]);
}

int dev_depth(Lane& L, const int16_t* disp16, int W, int H, const double* Q, float* depth) {
    if (Q) {
        QMat q;
        memcpy(q.q, Q, sizeof(q.q));
        L3D_LAUNCH(L, depth_q_kernel, dim3(cdiv(W, 128), H), 128, 0, disp16, W, H, q, depth);
    } else {
        size_t n = (size_t)W * H;
        L3D_LAUNCH(L, depth_default_kernel, cdiv(n, 256), 256, 0, disp16, n, depth);
    }
    return L3D_OK;
}

}  // namespace l3d
