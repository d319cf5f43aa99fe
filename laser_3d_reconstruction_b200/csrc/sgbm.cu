// sgbm.cu -- cv2.StereoSGBM.compute on sm_100a (modes SGBM / HH / SGBM_3WAY / HH4), bit-exact.
//
// Replaces stereo_matcher.compute / right_matcher.compute of the reference
// (camera/single_usb_stereo_camera.py:252-274 parameters, :324-325 calls).
//
// HBM layout: cost volume C and aggregated volume S are int16 [vrow][x][d] (d fastest), x in
// width1 = maxX1-minX1 coordinates.  A warp owns one pixel's disparity range: lane l holds DPL
// consecutive disparities packed as u16x2 words (DPL = 2/4/8/16 for D <= 64/128/256/512), so one warp
// access is one contiguous 64..1024 B segment.
//
// Kernels:
//   sgbm_prefilter_kernel     x-Sobel clip + half-pixel min/max, as pixel-pair operand entries (2 planes x 16 B / pixel)
//   sgbm_cost_dual_kernel     Birchfield-Tomasi pixel cost -> blockSize^2 box sum -> C (+P2) at block 5 / D 64,
//                             block 9 / D 128, block 11 / D 256: one volume (SGBM_3WAY's striped ones too, except at
//                             block 11 / D 256) or both matchers' single-segment volumes of a frame
//   sgbm_cost_kernel          the block-synchronous form: every other geometry, SGBM_3WAY's at block 11 / D 256 among them
//   sgbm_scan_hpair_kernel    both horizontal paths of a row in one CTA
//   sgbm_scan_kernel          one SGM path direction per launch, one warp per scan line, path state in registers,
//                             DPX u16x2 min/add, warp-wide min via CREDUX, C/S streamed through a cp.async ring; the
//                             last path can run the WTA (SCAN_FINAL; modes SGBM / HH / HH4)
//   sgbm_vgroup_kernel        (sgbm_vgroup.cu) the three previous-row paths of a pass fused on a thread-block cluster
//   sgbm_wta_lean_kernel      WTA + uniqueness + disp2 (atomicMax key) + sub-pixel, 32 pixels per warp (modes SGBM / HH / HH4)
//   sgbm_wta_lean3_kernel     the same walk with SGBM_3WAY's rules
//   sgbm_lrcheck_kernel       left-right consistency
// Value domain (see DESIGN.md): 0 <= L,S <= 32767 and C >= P2, which holds whenever the block sum
// does not wrap int16 (always for blockSize <= 9; for 11 unless every pixel of a block mismatches
// by more than 92 % of the maximum cost).  Inside that domain OpenCV's saturating int16 SIMD and
// the unsigned 16-bit arithmetic used here give identical bits.
#include <cuda_pipeline.h>

#include "sgbm.cuh"
#include "sgm_step.cuh"

namespace l3d {

constexpr unsigned FULL_MASK = 0xffffffffu;
constexpr uint32_t INF2 = 0x7fff7fffu;

int make_geom(const l3d_sgbm_params& p, int W, int H, Geom& g, std::string* err) {
    g.W = W; g.H = H; g.minD = p.minDisparity; g.D = p.numDisparities; g.maxD = g.minD + g.D;
    g.mode = p.mode;
    if (W < 2 || H < 1) { set_err(err, "sgbm: image too small"); return L3D_ERR_ARG; }
    if (g.D < 16 || g.D > 512 || (g.D % 16)) {
        set_err(err, "sgbm: numDisparities must be a multiple of 16 in [16,512], got %d", g.D);
        return L3D_ERR_UNSUPPORTED;
    }
    if (p.blockSize < 1 || !(p.blockSize & 1) || p.blockSize > 21) {
        set_err(err, "sgbm: blockSize must be odd in [1,21], got %d", p.blockSize);
        return L3D_ERR_UNSUPPORTED;
    }
    // Above 272 disparities the block-synchronous cost kernel's row-sum ring leaves room for tiles of 16 computed
    // columns only (sgbm_cost_single), and a tile must be wider than the window's 2 * (blockSize / 2) halo columns.
    if (g.D > 272 && p.blockSize > 15) {
        set_err(err, "sgbm: blockSize %d with numDisparities %d unsupported (blockSize <= 15 above 272 disparities)",
                p.blockSize, g.D);
        return L3D_ERR_UNSUPPORTED;
    }
    if (p.mode < 0 || p.mode > 3) { set_err(err, "sgbm: mode %d unsupported (0 SGBM, 1 HH, 2 SGBM_3WAY, 3 HH4)", p.mode); return L3D_ERR_UNSUPPORTED; }
    g.bs = p.blockSize; g.SW2 = p.blockSize / 2;
    g.uniq = p.uniquenessRatio >= 0 ? p.uniquenessRatio : 10;
    g.d12 = p.disp12MaxDiff > 0 ? p.disp12MaxDiff : 1;
    g.P1 = p.P1 > 0 ? p.P1 : 2;
    g.P2 = std::max(p.P2 > 0 ? p.P2 : 5, g.P1 + 1);
    if (g.P2 > 16000) { set_err(err, "sgbm: P2=%d exceeds the int16 value domain", g.P2); return L3D_ERR_UNSUPPORTED; }
    g.ftzero = std::max(p.preFilterCap, 15) | 1;
    if (g.ftzero > 127) { set_err(err, "sgbm: preFilterCap too large"); return L3D_ERR_UNSUPPORTED; }
    // the cost kernel adds u16x2 pairs with plain 32-bit arithmetic: every C value must fit 16 bits
    if (g.P2 + g.bs * g.bs * (2 * g.ftzero + 63) > 65535) {
        set_err(err, "sgbm: P2=%d with blockSize=%d exceeds the 16-bit cost domain", g.P2, g.bs);
        return L3D_ERR_UNSUPPORTED;
    }
    g.minX1 = std::max(g.maxD, 0); g.maxX1 = W + std::min(g.minD, 0); g.width1 = sgbm_width1(p, W);
    g.DPL = g.D <= 64 ? 2 : (g.D <= 128 ? 4 : (g.D <= 256 ? 8 : 16));
    g.NP = g.DPL / 2;
    g.nact = g.D / g.DPL;
    if (g.mode == 2) {
        const int nstripes = 4;
        int stripe_sz = (H + nstripes - 1) / nstripes;
        double t = 0.1 * stripe_sz; int ci = (int)t; if ((double)ci < t) ci++;
        int overlap = (g.bs / 2 + 1) + ci;
        g.nseg = 0; g.HV = 0;
        for (int s = 0; s < MAXSEG; s++) g.seg_shift[s] = 0;
        for (int s = 0; s < nstripes; s++) {
            int y0 = std::max(std::min(s * stripe_sz - overlap, H), 0);
            int y1 = std::min((s + 1) * stripe_sz, H);
            if (y1 <= y0) continue;
            int i = g.nseg++;
            g.seg_vr0[i] = g.HV; g.seg_y0[i] = y0; g.seg_rows[i] = y1 - y0; g.seg_emit[i] = s * stripe_sz;
            // OpenCV keeps every stripe in a buffer of its own (image row y at buffer row (s == 0 ? overlap : 0) + y - y0)
            // and assembles output row i from buffer row overlap + i % stripe_sz of stripe i / stripe_sz.  Where the stripe
            // start is clamped at the image top (s >= 1, s * stripe_sz < overlap: images of a few rows) the two do not meet:
            // output row i shows the result of image row i + shift and the rows past the stripe end stay invalid.  Found by
            // differential fuzzing of the oracle against cv2; restated in oracle/csrc/orc_sgbm.c.
            g.seg_shift[i] = s >= 1 ? std::max(overlap - s * stripe_sz, 0) : 0;
            g.HV += y1 - y0;
        }
    } else {
        g.nseg = 1; g.HV = H;
        g.seg_vr0[0] = 0; g.seg_y0[0] = 0; g.seg_rows[0] = H; g.seg_emit[0] = 0;
        for (int s = 0; s < MAXSEG; s++) g.seg_shift[s] = 0;
    }
    return L3D_OK;
}

int sgbm_volume_rows(const l3d_sgbm_params& p, int W, int H) {
    Geom g; std::string e;
    if (make_geom(p, W, H, g, &e) != L3D_OK) return -1;
    return g.HV;
}

// ------------------------------------------------------------------------------------------
// directional aggregation scan
// ------------------------------------------------------------------------------------------
// The kernels take ScanArgs and WtaArgs as __grid_constant__: they index the segment tables at run time, and NVVM copies
// a by-value parameter of up to 128 bytes (the size of both) into a local-memory stack frame to do that unless the
// parameter is declared read-only.
struct ScanArgs {
    const int16_t* C; int16_t* S;
    int width1, D, nact, P1, P2;
    uint32_t zero;  // 0, as a value the compiler cannot see (sgm_step.cuh)
    int hp_row0;    // horizontal pair: first volume row of this launch (row waves)
    int kind;   // 0 ->, 1 <-, 2 down, 3 down-right, 4 down-left, 5 up, 6 up-left, 7 up-right
    int store;  // 1: S = L ; 0: S = min(S + L, 32767)
    int HV, nseg;
    int lines_per_seg;  // kinds >= 2: lines per segment (columns, or diagonals)
    int seg_vr0[MAXSEG], seg_rows[MAXSEG];
    // SCAN_FINAL only: the winner-takes-all stage fused into the last path (modes SGBM / HH / HH4: one segment)
    int16_t* raw; unsigned* disp2key;
    int W, minD, minX1, uniq;
};
enum { SCAN_STORE = 0, SCAN_ACCUM = 1, SCAN_FINAL = 2 };  // S = L | S = sat(S + L) | sat(S + L) -> WTA, S not written

template <int NP> struct VecOf;
template <> struct VecOf<1> { typedef uint32_t T; };
template <> struct VecOf<2> { typedef uint2 T; };
template <> struct VecOf<4> { typedef uint4 T; };
struct __align__(32) u32x8 { uint4 lo, hi; };   // D in (256, 512]: 16 disparities per lane
template <> struct VecOf<8> { typedef u32x8 T; };

template <int NP> __device__ __forceinline__ void vec_unpack(const typename VecOf<NP>::T& v, uint32_t (&o)[NP]);
template <> __device__ __forceinline__ void vec_unpack<1>(const uint32_t& v, uint32_t (&o)[1]) { o[0] = v; }
template <> __device__ __forceinline__ void vec_unpack<2>(const uint2& v, uint32_t (&o)[2]) { o[0] = v.x; o[1] = v.y; }
template <> __device__ __forceinline__ void vec_unpack<4>(const uint4& v, uint32_t (&o)[4]) { o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w; }
template <> __device__ __forceinline__ void vec_unpack<8>(const u32x8& v, uint32_t (&o)[8]) {
    o[0] = v.lo.x; o[1] = v.lo.y; o[2] = v.lo.z; o[3] = v.lo.w; o[4] = v.hi.x; o[5] = v.hi.y; o[6] = v.hi.z; o[7] = v.hi.w;
}
template <int NP> __device__ __forceinline__ typename VecOf<NP>::T vec_pack(const uint32_t (&o)[NP]);
template <> __device__ __forceinline__ uint32_t vec_pack<1>(const uint32_t (&o)[1]) { return o[0]; }
template <> __device__ __forceinline__ uint2 vec_pack<2>(const uint32_t (&o)[2]) { return make_uint2(o[0], o[1]); }
template <> __device__ __forceinline__ uint4 vec_pack<4>(const uint32_t (&o)[4]) { return make_uint4(o[0], o[1], o[2], o[3]); }
template <> __device__ __forceinline__ u32x8 vec_pack<8>(const uint32_t (&o)[8]) {
    return u32x8{make_uint4(o[0], o[1], o[2], o[3]), make_uint4(o[4], o[5], o[6], o[7])};
}
// read-only global load of one lane's words (the lean WTA kernels).  NP = 8 takes two 16-byte loads: one 32-byte
// access (ld.global.nc.v8.b32) was measured too and was no faster (MODE_HH pipeline at 1920x1080 / D 384: 57.1 against
// 58.0 frames/s, with 32-byte S stores in the scans as well)
template <int NP> __device__ __forceinline__ typename VecOf<NP>::T vec_ldg(const typename VecOf<NP>::T* p) { return __ldg(p); }
template <> __device__ __forceinline__ u32x8 vec_ldg<8>(const u32x8* p) {
    return u32x8{__ldg(&p->lo), __ldg(&p->hi)};
}

constexpr int SCAN_WARPS = 4;

// Scan lines of one path direction.  kinds: 0 ->, 1 <-, 2 down, 3 down-right, 4 down-left, 5 up,
// 6 up-left, 7 up-right (direction of travel; the predecessor is one step behind).  Horizontal
// and vertical lines are rows / columns; the diagonal kinds run over true (anti-)diagonals of
// varying length, so there is no wrap-around logic in the loop.
struct ScanLine { int vr, x, n, dvr, dx; };

__device__ __forceinline__ bool scan_decode(const ScanArgs& a, int line, ScanLine& o) {
    const int width1 = a.width1, kind = a.kind;
    if (kind <= 1) {
        if (line >= a.HV) return false;
        o.vr = line; o.n = width1; o.dvr = 0;
        if (kind == 0) { o.x = 0; o.dx = 1; } else { o.x = width1 - 1; o.dx = -1; }
        return true;
    }
    const int lps = a.lines_per_seg;
    const int seg = line / lps, u = line - seg * lps;
    if (seg >= a.nseg) return false;
    const int rows = a.seg_rows[seg], top = a.seg_vr0[seg];
    int y0, x0, n;
    if (kind == 2 || kind == 5) {
        if (u >= width1) return false;
        y0 = 0; x0 = u; n = rows;
        o.dx = 0;
    } else if (kind == 3 || kind == 6) {  // diagonals x - y = u - (rows - 1)
        const int uu = u - (rows - 1);
        if (uu > width1 - 1) return false;
        y0 = max(0, -uu); x0 = uu + y0; n = min(rows - y0, width1 - x0);
        o.dx = 1;
    } else {  // anti-diagonals x + y = u
        if (u > width1 + rows - 2) return false;
        y0 = max(0, u - (width1 - 1)); x0 = u - y0; n = min(rows - y0, x0 + 1);
        o.dx = -1;
    }
    o.dvr = 1;
    if (kind >= 5) {  // bottom-up: start from the other end of the same line
        y0 += n - 1; x0 += o.dx * (n - 1);
        o.dvr = -1; o.dx = -o.dx;
    }
    o.vr = top + y0; o.x = x0; o.n = n;
    return n > 0;
}

// ---- async copy helpers ------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Winner-takes-all key: (cost << KS) | d, so that one unsigned minimum finds the lowest cost and, among equal costs, the
// first disparity.  d needs 8 bits up to D = 256 and 9 bits above; the cost (<= 32767) takes 15.
template <int NP> __host__ __device__ constexpr int wta_kshift() { return NP == 8 ? 9 : 8; }
template <int NP> __host__ __device__ constexpr unsigned wta_dmask() { return (1u << wta_kshift<NP>()) - 1u; }
// the keys of both halves of a packed u16x2 word whose low half holds disparity d0
template <int NP> __device__ __forceinline__ unsigned wta_key_lo(uint32_t w, unsigned d0) {
    constexpr int KS = wta_kshift<NP>();
    return ((w << KS) & (0xffffu << KS)) | d0;
}
template <int NP> __device__ __forceinline__ unsigned wta_key_hi(uint32_t w, unsigned d0) {
    constexpr int KS = wta_kshift<NP>();
    return ((w >> (16 - KS)) & (0xffffu << KS)) | (d0 + 1);
}

// OpenCV's uniqueness test (modes SGBM / HH): reject when another disparity further than 1 from
// the winner costs less than minS * 100 / (100 - uniq).  Kept out of line: only the as-constructed
// parameter set (uniquenessRatio > 0) pays for it.
template <int NP>
__device__ __noinline__ bool wta_not_unique(const uint32_t (&w)[NP], unsigned key, int uniq, unsigned dkey, bool active) {
    const int minS = (int)(key >> wta_kshift<NP>()), best = (int)(key & wta_dmask<NP>());
    bool rej = false;
#pragma unroll
    for (int q = 0; q < NP; q++) {
        const int s0 = (int)(w[q] & 0xffffu), s1 = (int)(w[q] >> 16);
        const int d0 = (int)dkey + 2 * q;
        if (active && s0 * (100 - uniq) < minS * 100 && abs(best - d0) > 1) rej = true;
        if (active && s1 * (100 - uniq) < minS * 100 && abs(best - d0 - 1) > 1) rej = true;
    }
    return __any_sync(FULL_MASK, rej) && minS < 32767;
}

// cp.async ring of the scan kernels, per words per lane
template <int NP> struct ScanRing {
    static constexpr int CH = 16;     // steps per chunk (divides 32: SCAN_FINAL flushes its WTA every 32 steps)
    static constexpr int NST = 3;     // chunks in flight per warp (two chunks = 32 steps of look-ahead)
    static constexpr int HP_NST = 2;  // horizontal pair: 1440 warps must be resident at once, a shallower ring keeps the launch to one wave
};
// D in (256, 512]: a step moves 512..1024 bytes per array and has twice the arithmetic of D = 256; a ring of two 8-step
// chunks half the size lets twice the one-warp CTAs share an SM (SCAN_FINAL at D = 384: 49 KB instead of 98 KB), which
// is worth more than the deeper look-ahead.  1920x1080 / D 384 / block 11 on a B200, kernels alone: SCAN_FINAL 1.737 -> 0.760 ms, accumulating scans
// 0.64-0.72 -> 0.63-0.70 ms, horizontal pair 0.95 -> 1.00 ms; MODE_HH pipeline 58.0 -> 68.8 frames/s (4 lanes).
// Also measured: 8 x 3 (66.5 frames/s), 4 x 4 (67.5), 4 x 3 (68.2).
template <> struct ScanRing<8> {
    static constexpr int CH = 8;
    static constexpr int NST = 2;
    static constexpr int HP_NST = 2;
};
template <int NP> __device__ __host__ __forceinline__ size_t scan_smem_bytes_dev(int D) {
    return (size_t)ScanRing<NP>::HP_NST * ScanRing<NP>::CH * (D * 2) * 2;
}
template <int NP> static size_t scan_smem_bytes(int D, int smode) {
    return (size_t)ScanRing<NP>::NST * ScanRing<NP>::CH * (D * 2) * (smode == 0 ? 1 : 2) + (smode == 2 ? (size_t)32 * D * 2 : 0);
}

// One warp (= one CTA) per scan line.  The line's C (and, when accumulating, S) vectors are staged
// through a shared-memory ring with 16-byte cp.async copies (LDGSTS.128: one instruction moves 512
// contiguous ring bytes = two 128-disparity steps), NST - 1 chunks of ScanRing<NP>::CH steps ahead of the
// consumer (32 steps for NP <= 4, 8 for NP = 8), so that the HBM latency is off the recurrence's critical
// path; the recurrence itself lives in registers.
template <int NP, int SMODE, bool FULL, int NST>
__device__ __forceinline__ void scan_run(const ScanArgs& a, const ScanLine& ln, unsigned char* scan_smem,
                                         uint32_t (&L)[NP], uint32_t& minL, const int lane) {
    typedef typename VecOf<NP>::T vec;
    constexpr int CH = ScanRing<NP>::CH;
    constexpr bool STORE = SMODE == SCAN_STORE;
    constexpr bool FINAL = SMODE == SCAN_FINAL;
    constexpr int DPL = NP * 2;
    const int nact = a.nact, n = ln.n;
    const bool active = FULL || lane < nact;
    const uint32_t B = (uint32_t)a.D * 2u;                      // bytes per pixel vector
    const uint32_t stage_bytes = CH * B * (STORE ? 1 : 2);
    const uint32_t ring = smem_u32(scan_smem);
    const long pstride = (long)ln.dvr * a.width1 + ln.dx;      // pixel-index step along the line
    const long pix0 = (long)ln.vr * a.width1 + ln.x;
    const char* __restrict__ Cb = (const char*)a.C;
    const char* __restrict__ Sb = (const char*)a.S;
    vec* __restrict__ Sv = (vec*)a.S;
    const int nchunks = (n + CH - 1) / CH;
    // 16-byte pieces: ppv per pixel vector, CH * ppv per chunk and array; piece p = it * 32 + lane
    const int ppv = a.D >> 3;
    const int pieces = CH * ppv;
    const int li0 = lane / ppv, lr0 = lane - li0 * ppv, di = 32 / ppv, dr = 32 - di * ppv;
    const long step_bytes = pstride * (long)B;                      // between consecutive steps of the line
    const long it_bytes = (long)di * step_bytes + (long)dr * 16;    // piece p -> p + 32
    const long wrap_bytes = step_bytes - (long)ppv * 16;            // extra when the piece index wraps into the next step
    const long lane_off = pix0 * (long)B + (long)li0 * step_bytes + (long)lr0 * 16;
    auto issue = [&](int chunk) {
        if (chunk < nchunks) {
            const int first = chunk * CH;
            const int cnt = min(CH, n - first);
            uint32_t dst = ring + (chunk % NST) * stage_bytes + lane * 16;
            long off = lane_off + (long)first * step_bytes;
            if constexpr (FULL && 8 * NP > 32) {
                // D = 512: a pixel vector is 64 pieces, two warp-wide iterations of 32 pieces per step
                constexpr int SPI = 8 * NP / 32, ITERS = CH * SPI;
#pragma unroll
                for (int it = 0; it < ITERS; it++) {
                    if (cnt == CH || it / SPI < cnt) {
                        const long o = off + (long)(it / SPI) * step_bytes + (it % SPI) * 512;
                        cp_async16(dst + it * 512, Cb + o);
                        if (!STORE) cp_async16(dst + it * 512 + CH * B, Sb + o);
                    }
                }
            } else if (FULL) {
                // D = 64 * NP: a pixel vector is 8 * NP pieces, which divides 32 -- no piece straddles two
                // steps' boundaries differently per iteration, every constant folds
                constexpr int PPV = 8 * NP, DI = 32 / PPV, ITERS = CH * PPV / 32;
                const long it_b = (long)DI * step_bytes;
                if (cnt == CH) {
#pragma unroll
                    for (int it = 0; it < ITERS; it++) {
                        cp_async16(dst + it * 512, Cb + off);
                        if (!STORE) cp_async16(dst + it * 512 + CH * B, Sb + off);
                        off += it_b;
                    }
                } else {
#pragma unroll
                    for (int it = 0; it < ITERS; it++) {
                        if (li0 + it * DI < cnt) {
                            cp_async16(dst + it * 512, Cb + off);
                            if (!STORE) cp_async16(dst + it * 512 + CH * B, Sb + off);
                        }
                        off += it_b;
                    }
                }
            } else {
                int i = li0, r = lr0;
                for (int p = lane; p < pieces; p += 32) {
                    if (i < cnt) {
                        cp_async16(dst, Cb + off);
                        if (!STORE) cp_async16(dst + CH * B, Sb + off);
                    }
                    dst += 512; i += di; r += dr; off += it_bytes;
                    if (r >= ppv) { r -= ppv; i++; off += wrap_bytes; }
                }
            }
        }
        cp_async_commit();
    };
#pragma unroll
    for (int c = 0; c < NST; c++) issue(c);

    const uint32_t p1x2 = (uint32_t)a.P1 * 0x10001u;
    const uint32_t k2 = (0x10000u - (uint32_t)a.P2) * 0x10001u;
    const SgmLane sl = sgm_lane_init(lane, a.zero);
    const int vstride = (int)pstride * nact;                    // vec-index step
    unsigned so = (unsigned)pix0 * (unsigned)nact + (unsigned)lane;

    // SCAN_FINAL: the finished S vectors of the last (up to) 32 steps are stashed in shared memory and
    // their arg-min keys parked one per lane; every 32 steps lane k finishes pixel k (disp2 vote,
    // sub-pixel interpolation with its integer division, store) -- once per 32 pixels, in parallel.
    unsigned wkey = 0xffffffffu;
    bool wrej = false;
    int nsteps = 0;  // steps done so far (warp-uniform)
    const unsigned dkey = (unsigned)(lane * DPL);
    unsigned char* stash = scan_smem + NST * stage_bytes;  // [32][B]
    auto wta_flush = [&](int first_step, int count) {
        __syncwarp();
        const int minS = (int)(wkey >> wta_kshift<NP>()), d = (int)(wkey & wta_dmask<NP>());
        const int j = first_step + lane;
        const int y = ln.vr + ln.dvr * j;
        const int x = ln.x + ln.dx * j;
        if (lane < count && !wrej && minS < 32767) {  // minS == 32767: nothing beat MAX_COST, pixel stays invalid
            const int x2 = x + a.minX1 - d - a.minD;
            if (x2 >= 0 && x2 < a.W + 2)
                atomicMax(a.disp2key + (size_t)y * (a.W + 2) + x2, ((unsigned)(0x7fff - minS) << 16) | (unsigned)x);
            int dd = d * 16;
            if (0 < d && d < a.D - 1) {
                const uint16_t* Sp = (const uint16_t*)(stash + (size_t)lane * B);
                const int sm = Sp[d - 1], sp = Sp[d + 1];
                const int denom2 = max(sm + sp - 2 * minS, 1);
                dd += ((sm - sp) * 16 + denom2) / (denom2 * 2);
            }
            a.raw[(size_t)y * a.W + x + a.minX1] = (int16_t)(dd + a.minD * 16);
        }
        wrej = false;
        __syncwarp();
    };
    auto step = [&](const vec* cs, const vec* ss, int i) {
        uint32_t Cw[NP], Sw[NP];
        if (active) {
            vec_unpack<NP>(cs[i * nact + lane], Cw);
            if (!STORE) vec_unpack<NP>(ss[i * nact + lane], Sw);
        } else {
#pragma unroll
            for (int q = 0; q < NP; q++) { Cw[q] = 0; Sw[q] = 0; }
        }
        minL = sgm_step<NP, false, FULL>(L, L, minL, Cw, p1x2, k2, sl, active);
        uint32_t out[NP];
#pragma unroll
        for (int q = 0; q < NP; q++) out[q] = STORE ? L[q] : __viaddmin_u16x2(Sw[q], L[q], INF2);
        if (!FINAL) {
            if (active) Sv[so] = vec_pack<NP>(out);
            so += (unsigned)vstride;
        } else {
            // winner-takes-all on the finished S vector (first minimum wins, as OpenCV's strict '<')
            if (!FULL && !active) {
#pragma unroll
                for (int q = 0; q < NP; q++) out[q] = INF2;
            }
            unsigned key = 0xffffffffu;
            bool rej = false;
            const int slot = nsteps & 31;
            if (active) *(vec*)(stash + (size_t)slot * B + (size_t)lane * sizeof(vec)) = vec_pack<NP>(out);
#pragma unroll
            for (int q = 0; q < NP; q++) {
                key = min(key, wta_key_lo<NP>(out[q], dkey + 2 * q));
                key = min(key, wta_key_hi<NP>(out[q], dkey + 2 * q));
            }
            key = __reduce_min_sync(FULL_MASK, key);
            if (a.uniq > 0) rej = wta_not_unique<NP>(out, key, a.uniq, dkey, active);
            if (lane == slot) { wkey = key; wrej = rej; }
            nsteps++;
        }
    };
    for (int c = 0; c < nchunks; c++) {
        const int s = c % NST;
        cp_async_wait<NST - 1>();
        __syncwarp();
        const vec* cs = (const vec*)(scan_smem + s * stage_bytes);
        const vec* ss = (const vec*)(scan_smem + s * stage_bytes + CH * B);
        const int cnt = min(CH, n - c * CH);
        if (cnt == CH) {
#pragma unroll
            for (int i = 0; i < CH; i++) step(cs, ss, i);
        } else {
            for (int i = 0; i < cnt; i++) step(cs, ss, i);
        }
        __syncwarp();  // every lane is done reading the slot before it is refilled
        issue(c + NST);
        if (FINAL && (nsteps & 31) == 0) wta_flush(nsteps - 32, 32);  // CH divides 32
    }
    if (FINAL && (nsteps & 31)) wta_flush(nsteps & ~31, nsteps & 31);
}

template <int NP, int SMODE, bool FULL>
__global__ void __launch_bounds__(32) sgbm_scan_kernel(const __grid_constant__ ScanArgs a) {
    extern __shared__ __align__(128) unsigned char scan_smem[];
    const int lane = threadIdx.x;
    ScanLine ln;
    if (!scan_decode(a, blockIdx.x, ln)) return;
    uint32_t L[NP];
#pragma unroll
    for (int k = 0; k < NP; k++) L[k] = (FULL || lane < a.nact) ? 0u : INF2;
    uint32_t minL = 0;  // packed: warp-wide min of L in both halves
    scan_run<NP, SMODE, FULL, ScanRing<NP>::NST>(a, ln, scan_smem, L, minL, lane);
}

// Both horizontal paths of one row in one CTA of two warps: warp 0 runs left-to-right, warp 1
// right-to-left.  Each first covers its own half storing S = L; at the middle the two exchange
// their path states and each walks back over its own half with the other direction's path,
// accumulating S = sat(S + L) -- every S vector is written once and read-modified once, and the
// two serial recurrences of a row run concurrently.
template <int NP, bool FULL>
__global__ void __launch_bounds__(64) sgbm_scan_hpair_kernel(const __grid_constant__ ScanArgs a) {
    extern __shared__ __align__(128) unsigned char scan_smem[];
    __shared__ uint32_t xch[2][32][NP + 1];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    unsigned char* my_smem = scan_smem + (size_t)warp * scan_smem_bytes_dev<NP>(a.D);
    const int vr = a.hp_row0 + blockIdx.x, width1 = a.width1, mid = width1 / 2;
    ScanLine s1, s2;
    s1.vr = s2.vr = vr; s1.dvr = s2.dvr = 0;
    if (warp == 0) { s1.x = 0; s1.n = mid; s1.dx = 1; s2.x = mid - 1; s2.n = mid; s2.dx = -1; }
    else { s1.x = width1 - 1; s1.n = width1 - mid; s1.dx = -1; s2.x = mid; s2.n = width1 - mid; s2.dx = 1; }
    uint32_t L[NP];
#pragma unroll
    for (int k = 0; k < NP; k++) L[k] = (FULL || lane < a.nact) ? 0u : INF2;
    uint32_t minL = 0;
    scan_run<NP, SCAN_STORE, FULL, ScanRing<NP>::HP_NST>(a, s1, my_smem, L, minL, lane);
    // turn round: the two warps exchange their path states at the middle and each walks back over ITS OWN half with
    // the other direction's path -- the vectors it needs first are the ones it touched last (L2 reuse distance grows
    // from zero instead of being half a row for every vector)
#pragma unroll
    for (int k = 0; k < NP; k++) xch[warp][lane][k] = L[k];
    xch[warp][lane][NP] = minL;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < NP; k++) L[k] = xch[warp ^ 1][lane][k];
    minL = xch[warp ^ 1][lane][NP];
    scan_run<NP, SCAN_ACCUM, FULL, ScanRing<NP>::HP_NST>(a, s2, my_smem, L, minL, lane);
}

// ------------------------------------------------------------------------------------------
// WTA + uniqueness + disp2 + sub-pixel
// ------------------------------------------------------------------------------------------
struct WtaArgs {
    const int16_t* S; int16_t* raw; unsigned* disp2key;
    int W, width1, D, nact, DPL, minD, minX1, uniq;
    int HV, nseg;
    int seg_vr0[MAXSEG], seg_y0[MAXSEG], seg_rows[MAXSEG], seg_emit[MAXSEG];
};
constexpr int WTA_WARPS = 8;

// Lean WTA for modes SGBM / HH (single segment): a warp walks 32 consecutive pixels; for each it
// loads the pixel's S vector (one coalesced 64..512 B access), reduces a packed (cost << 8 | d) key
// with CREDUX (first minimum wins, as OpenCV's strict '<' scan) and parks the result in lane k.
// The per-pixel tail (disp2 vote, sub-pixel interpolation with its integer division, store) then
// runs once for 32 pixels in parallel instead of once per pixel on one lane.
template <int NP, bool FULL>
__global__ void __launch_bounds__(WTA_WARPS * 32) sgbm_wta_lean_kernel(const __grid_constant__ WtaArgs a) {
    typedef typename VecOf<NP>::T vec;
    constexpr int DPL = NP * 2;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long npix = (long)a.HV * a.width1;
    const long base = ((long)blockIdx.x * WTA_WARPS + warp) * 32;
    if (base >= npix) return;
    const int cnt = (int)min(32L, npix - base);
    const int nact = a.nact;
    const bool active = FULL || lane < nact;
    const vec* __restrict__ Sv = (const vec*)a.S + (size_t)base * nact + lane;
    const unsigned dkey = (unsigned)(lane * DPL);
    const int uniq = a.uniq;
    unsigned mykey = 0xffffffffu;
    bool myok = false;
    for (int k = 0; k < cnt; k++) {
        uint32_t w[NP];
        if (active) vec_unpack<NP>(vec_ldg<NP>(Sv + (size_t)k * nact), w);
        else {
#pragma unroll
            for (int q = 0; q < NP; q++) w[q] = INF2;
        }
        unsigned key = 0xffffffffu;
#pragma unroll
        for (int q = 0; q < NP; q++) {
            key = min(key, wta_key_lo<NP>(w[q], dkey + 2 * q));
            key = min(key, wta_key_hi<NP>(w[q], dkey + 2 * q));
        }
        key = __reduce_min_sync(FULL_MASK, key);
        const int minS = (int)(key >> wta_kshift<NP>()), best = (int)(key & wta_dmask<NP>());
        bool ok = minS < 32767;  // nothing beats MAX_COST: pixel stays invalid, disp2 untouched
        if (uniq > 0 && ok) {
            bool rej = false;
#pragma unroll
            for (int q = 0; q < NP; q++) {
                const int s0 = (int)(w[q] & 0xffffu), s1 = (int)(w[q] >> 16);
                const int d0 = (int)dkey + 2 * q;
                if (active && s0 * (100 - uniq) < minS * 100 && abs(best - d0) > 1) rej = true;
                if (active && s1 * (100 - uniq) < minS * 100 && abs(best - d0 - 1) > 1) rej = true;
            }
            ok = !__any_sync(FULL_MASK, rej);
        }
        if (lane == k) { mykey = key; myok = ok; }
    }
    if (lane < cnt && myok) {
        const long pix = base + lane;
        const int y = (int)(pix / a.width1), x = (int)(pix - (long)y * a.width1);
        const int minS = (int)(mykey >> wta_kshift<NP>()), d = (int)(mykey & wta_dmask<NP>());
        const int x2 = x + a.minX1 - d - a.minD;
        if (x2 >= 0 && x2 < a.W + 2)
            atomicMax(a.disp2key + (size_t)y * (a.W + 2) + x2, ((unsigned)(0x7fff - minS) << 16) | (unsigned)x);
        int dd = d * 16;
        if (0 < d && d < a.D - 1) {
            const int16_t* Sp = a.S + (size_t)pix * a.D;
            const int sm = Sp[d - 1], sp = Sp[d + 1];
            const int denom2 = max(sm + sp - 2 * minS, 1);
            dd += ((sm - sp) * 16 + denom2) / (denom2 * 2);
        }
        a.raw[(size_t)y * a.W + x + a.minX1] = (int16_t)(dd + a.minD * 16);
    }
}

// Lean WTA for mode SGBM_3WAY: the same 32-pixels-per-warp walk over the stripe volumes, with that mode's rules (the
// 8-lane SIMD arg-min, the SIMD form of the uniqueness test, disp2 votes only inside [0, W), overlap rows of a stripe
// not emitted).
template <int NP>
__global__ void __launch_bounds__(WTA_WARPS * 32) sgbm_wta_lean3_kernel(const __grid_constant__ WtaArgs a) {
    typedef typename VecOf<NP>::T vec;
    constexpr int DPL = NP * 2;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int width1 = a.width1;
    const long npix = (long)a.HV * width1;
    const long base = ((long)blockIdx.x * WTA_WARPS + warp) * 32;
    if (base >= npix) return;
    const int cnt = (int)min(32L, npix - base);
    const int nact = a.nact;
    const bool active = lane < nact;
    // this lane's pixel (lane < cnt): volume row -> stripe -> image row; rows of a stripe's overlap are not emitted
    const long mypix = base + min(lane, cnt - 1);
    const int vr = (int)(mypix / width1), x = (int)(mypix - (long)vr * width1);
    int seg = 0;
    for (int q = 1; q < a.nseg; q++) if (vr >= a.seg_vr0[q]) seg = q;
    const int y = a.seg_y0[seg] + (vr - a.seg_vr0[seg]);
    const bool emit = lane < cnt && y >= a.seg_emit[seg];
    const unsigned emit_mask = __ballot_sync(FULL_MASK, emit);
    if (!emit_mask) return;
    const vec* __restrict__ Sv = (const vec*)a.S + (size_t)base * nact + lane;
    const int uniq = a.uniq;
    unsigned mykey = 0;
    bool myok = false;
    for (int k = 0; k < cnt; k++) {
        if (!((emit_mask >> k) & 1u)) continue;  // warp-uniform
        uint32_t w[NP];
        if (active) vec_unpack<NP>(vec_ldg<NP>(Sv + (size_t)k * nact), w);
        else {
#pragma unroll
            for (int q = 0; q < NP; q++) w[q] = INF2;
        }
        int sv[DPL];
#pragma unroll
        for (int q = 0; q < NP; q++) { sv[2 * q] = (int)(w[q] & 0xffffu); sv[2 * q + 1] = (int)(w[q] >> 16); }
        int m = 32767;
#pragma unroll
        for (int j = 0; j < DPL; j++) m = min(m, sv[j]);
        const int minS = __reduce_min_sync(FULL_MASK, m);
        // OpenCV's 8-lane SIMD arg-min: per residue class d mod 8 the LAST disparity that attains the minimum, then the
        // smallest of those.  One ballot per register slot j gives the lanes holding the minimum at d = lane * DPL + j;
        // the classes of a slot are lane patterns (d mod 8 = (lane * DPL + j) mod 8), so "last in class" is the highest
        // set bit of the ballot under the class's lane mask.  DPL 16: every lane holds two disparities of each class, at
        // slots c and c + 8; the last of class c is the larger of the two slots' highest candidates.
        int best = 0x7fffffff;
        if constexpr (DPL > 8) {
#pragma unroll
            for (int c = 0; c < 8; c++) {
                int last = -1;
#pragma unroll
                for (int j = c; j < DPL; j += 8) {
                    const unsigned b = __ballot_sync(FULL_MASK, active && sv[j] == minS);
                    if (b) last = max(last, (31 - __clz(b)) * DPL + j);
                }
                if (last >= 0) best = min(best, last);
            }
        } else {
#pragma unroll
            for (int j = 0; j < DPL; j++) {
                const unsigned b = __ballot_sync(FULL_MASK, active && sv[j] == minS);
                constexpr int LPC = 8 / DPL;                     // lanes per period of d mod 8 (DPL 2: 4, DPL 4: 2, DPL 8: 1)
#pragma unroll
                for (int r = 0; r < LPC; r++) {
                    unsigned pat = 0;                            // lanes with lane % LPC == r
#pragma unroll
                    for (int l = r; l < 32; l += LPC) pat |= 1u << l;
                    const unsigned mm = b & pat;
                    if (mm) best = min(best, (31 - __clz(mm)) * DPL + j);
                }
            }
        }
        bool ok = true;
        if (uniq > 0) {
            const int thresh = (100 * minS) / (100 - uniq);
            const int tr = (int)(short)(thresh + 1);
            bool rej = false;
#pragma unroll
            for (int j = 0; j < DPL; j++) {
                const int d = lane * DPL + j;
                if (active && sv[j] < tr && (d < best - 1 || d > best + 1)) rej = true;
            }
            ok = !__any_sync(FULL_MASK, rej);
        }
        if (lane == k) { mykey = ((unsigned)minS << wta_kshift<NP>()) | (unsigned)best; myok = ok; }
    }
    if (emit && myok) {
        const int minS = (int)(mykey >> wta_kshift<NP>()), d = (int)(mykey & wta_dmask<NP>());
        const int x2 = x + a.minX1 - d - a.minD;
        if (x2 >= 0 && x2 < a.W && minS < 32767)
            atomicMax(a.disp2key + (size_t)y * (a.W + 2) + x2, ((unsigned)(0x7fff - minS) << 16) | (unsigned)x);
        int dd = d * 16;
        if (0 < d && d < a.D - 1) {
            const int16_t* Sp = a.S + (size_t)mypix * a.D;
            const int sm = Sp[d - 1], sp = Sp[d + 1], sc = Sp[d];
            const int denom2 = max(sm + sp - 2 * sc, 1);
            dd += ((sm - sp) * 16 + denom2) / (denom2 * 2);
        }
        a.raw[(size_t)y * a.W + x + a.minX1] = (int16_t)(dd + a.minD * 16);
    }
}

__global__ void sgbm_lrcheck_kernel(int16_t* __restrict__ raw, const unsigned* __restrict__ disp2key, int W, int H,
                                    int minX1, int maxX1, int minD, int d12) {
    int x = minX1 + blockIdx.x * blockDim.x + threadIdx.x;
    int y = blockIdx.y;
    if (x >= maxX1) return;
    const int INVALID = (minD - 1) * 16;
    int d1 = raw[(size_t)y * W + x];
    if (d1 == INVALID) return;
    int _d = d1 >> 4, d_ = (d1 + 15) >> 4;
    int _x = x - _d, x_ = x - d_;
    const unsigned* k2 = disp2key + (size_t)y * (W + 2);
    bool c = true;
    if (0 <= _x && _x < W) {
        unsigned k = k2[_x];
        int d2 = (k >> 16) ? (int)(k & 0xffffu) + minX1 - _x : INVALID;  // unset entries hold the SCALED invalid value, as in OpenCV
        c = c && d2 >= minD && abs(d2 - _d) > d12;
    } else c = false;
    if (0 <= x_ && x_ < W) {
        unsigned k = k2[x_];
        int d2 = (k >> 16) ? (int)(k & 0xffffu) + minX1 - x_ : INVALID;
        c = c && d2 >= minD && abs(d2 - d_) > d12;
    } else c = false;
    if (c) raw[(size_t)y * W + x] = (int16_t)INVALID;
}

__global__ void fill_s16_kernel(int16_t* p, size_t n, int16_t v) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// ------------------------------------------------------------------------------------------
// host driver
// ------------------------------------------------------------------------------------------
template <int NP, int SMODE>
static int launch_scan_t(Lane& L, const ScanArgs& sa, int lines) {
    const size_t smem = scan_smem_bytes<NP>(sa.D, SMODE);
    if (sa.nact == 32) {
        L3D_CHECK(L, cudaFuncSetAttribute(sgbm_scan_kernel<NP, SMODE, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        L3D_LAUNCH(L, (sgbm_scan_kernel<NP, SMODE, true>), lines, 32, smem, sa);
    } else {
        L3D_CHECK(L, cudaFuncSetAttribute(sgbm_scan_kernel<NP, SMODE, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        L3D_LAUNCH(L, (sgbm_scan_kernel<NP, SMODE, false>), lines, 32, smem, sa);
    }
    return L3D_OK;
}
template <int NP>
static int launch_hpair(Lane& L, const ScanArgs& sa0) {
    const size_t smem = 2 * scan_smem_bytes_dev<NP>(sa0.D);
    // Row slices.  Alone, ONE launch over all rows is fastest (the two serial recurrences per row need every row in flight
    // to cover their latency: 0.168 ms against 0.213 ms in three slices at config 3) -- that is what single calls and the
    // kernel-timing leg use.  Inside the frame pipeline three slices let the other streams' kernels (above all the
    // aggregation clusters, which need whole free SMs) start sooner: +2 % frames/s (tools/skip_probe.py).
    const int hp_waves = (L.back_stream && !L.timing && sa0.HV >= 360) ? 3 : 1;
    ScanArgs sa = sa0;
    const int per = cdiv(sa.HV, hp_waves);
    for (int r0 = 0; r0 < sa.HV; r0 += per) {
        const int rows = std::min(per, sa.HV - r0);
        sa.hp_row0 = r0;
        if (sa.nact == 32) {
            L3D_CHECK(L, cudaFuncSetAttribute(sgbm_scan_hpair_kernel<NP, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            L3D_LAUNCH(L, (sgbm_scan_hpair_kernel<NP, true>), rows, 64, smem, sa);
        } else {
            L3D_CHECK(L, cudaFuncSetAttribute(sgbm_scan_hpair_kernel<NP, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            L3D_LAUNCH(L, (sgbm_scan_hpair_kernel<NP, false>), rows, 64, smem, sa);
        }
    }
    return L3D_OK;
}
template <int NP>
static int launch_scan_m(Lane& L, int smode, const ScanArgs& sa, int lines) {
    if (smode == SCAN_STORE) return launch_scan_t<NP, SCAN_STORE>(L, sa, lines);
    if (smode == SCAN_ACCUM) return launch_scan_t<NP, SCAN_ACCUM>(L, sa, lines);
    return launch_scan_t<NP, SCAN_FINAL>(L, sa, lines);
}
static int launch_scan_np(Lane& L, int NP, int smode, const ScanArgs& sa, int lines) {
    if (NP == 1) return launch_scan_m<1>(L, smode, sa, lines);
    if (NP == 2) return launch_scan_m<2>(L, smode, sa, lines);
    if (NP == 4) return launch_scan_m<4>(L, smode, sa, lines);
    return launch_scan_m<8>(L, smode, sa, lines);
}

// ------------------------------------------------------------------------------------------
// host driver.  One matcher run = front (descriptors, cost volume, both horizontal paths)
//                               + middle (the previous-row paths: cluster-fused or direction-split)
//                               + back (WTA if not fused, LR check, median, speckles).
// The frame pipeline runs the fronts of a group of frames on their lanes, ONE cluster-fused middle
// launch per pass over all the group's volumes, and the backs on the lanes again (pipeline.cu).
// ------------------------------------------------------------------------------------------

static void scan_args_of(const SgbmRun& r, ScanArgs& sa) {
    const Geom& g = r.g;
    sa.C = r.C; sa.S = r.S; sa.width1 = g.width1; sa.D = g.D; sa.nact = g.nact; sa.P1 = g.P1; sa.P2 = g.P2;
    sa.HV = g.HV; sa.nseg = g.nseg;
    for (int s = 0; s < MAXSEG; s++) { sa.seg_vr0[s] = g.seg_vr0[s]; sa.seg_rows[s] = g.seg_rows[s]; }
    sa.raw = r.raw; sa.disp2key = r.d2; sa.W = r.W; sa.minD = g.minD; sa.minX1 = g.minX1; sa.uniq = g.uniq;
    sa.kind = 0; sa.store = 1; sa.lines_per_seg = 0; sa.zero = 0; sa.hp_row0 = 0;
}

// front, first part: geometry, invalid-filled raw image, scratch volumes, disp2 vote buffer
// set: 0 / 1 selects the scratch slots (the pipeline keeps the left and the right matcher's volumes alive together)
static int sgbm_front_begin(Lane& L, const l3d_sgbm_params& p, int W, int H, int set, SgbmRun& r) {
    r.p = p; r.W = W; r.H = H; r.wta_done = false;  // r.no_hpair is the caller's choice and survives
    r.C = nullptr; r.S = nullptr; r.d2 = nullptr;
    Geom& g = r.g;
    int rc = make_geom(p, W, H, g, L.err);
    if (rc != L3D_OK) return rc;
    const size_t npix = (size_t)W * H;
    const int16_t INVALID = (int16_t)((g.minD - 1) * 16);
    r.raw = L.get<int16_t>(set ? S_RAW2 : S_RAW, npix);
    L3D_LAUNCH(L, fill_s16_kernel, cdiv(npix, 256), 256, 0, r.raw, npix, INVALID);
    if (g.width1 <= 0) return L3D_OK;
    const size_t nvol = (size_t)g.HV * g.width1 * g.D;
    r.C = L.get<int16_t>(set ? S_COST2 : S_COST, nvol);
    r.S = L.get<int16_t>(set ? S_AGGR2 : S_AGGR, nvol);
    const size_t nd2 = ((size_t)H * (W + 2) + 1) & ~(size_t)1;   // vote words, padded so that the records behind them are 8-byte aligned
    r.d2 = L.get<unsigned>(set ? S_DISP22 : S_DISP2, nd2 + 2 * (size_t)g.HV * g.width1);
    r.wrec = (uint2*)(r.d2 + nd2);
    L3D_CHECK(L, cudaMemsetAsync(r.d2, 0, (size_t)H * (W + 2) * sizeof(unsigned), L.stream));
    return L3D_OK;
}

// front, last part: MODE_HH4's constant bottom rows, then both horizontal paths of every row
static int sgbm_front_end(Lane& L, SgbmRun& r) {
    const Geom& g = r.g;
    const int H = r.H;
    if (g.width1 <= 0) return L3D_OK;
    if (g.mode == 3 && g.SW2 > 0 && H > 1) {
        // MODE_HH4: OpenCV's cost loop of this mode has no branch for window rows below the image, so the last
        // blockSize/2 rows of C (from row 1 on) keep their initial value P2 for every disparity (found by
        // differential testing against cv2 4.13, restated in oracle/csrc/orc_sgbm.c)
        const int y0 = std::max(H - g.SW2, 1);
        const size_t rowel = (size_t)g.width1 * g.D;
        L3D_LAUNCH(L, fill_s16_kernel, cdiv(rowel * (H - y0), 256), 256, 0, r.C + rowel * y0, rowel * (H - y0), (int16_t)g.P2);
    }
    if (r.no_hpair) return L3D_OK;
    ScanArgs sa;
    scan_args_of(r, sa);
    L.t_begin("sgbm_scan_k0");
    int rc = g.NP == 1 ? launch_hpair<1>(L, sa)
           : g.NP == 2 ? launch_hpair<2>(L, sa)
           : g.NP == 4 ? launch_hpair<4>(L, sa)
                       : launch_hpair<8>(L, sa);
    L.t_end("sgbm_scan_k0");
    return rc;
}

// descL/descR: BT operands of this run's left / right image, computed here when `make_desc`.
int sgbm_front(Lane& L, const l3d_sgbm_params& p, const uint8_t* left, const uint8_t* right, int W, int H, int set,
               uint4* dL, uint4* dR, bool make_desc, SgbmRun& r) {
    int rc = sgbm_front_begin(L, p, W, H, set, r);
    if (rc != L3D_OK) return rc;
    const Geom& g = r.g;
    if (g.width1 <= 0) return L3D_OK;
    if (make_desc) {
        if ((rc = sgbm_prefilter(L, left, W, H, g.ftzero, dL)) != L3D_OK) return rc;
        if ((rc = sgbm_prefilter(L, right, W, H, g.ftzero, dR)) != L3D_OK) return rc;
    }
    L.t_begin("sgbm_cost");
    rc = sgbm_cost_single(L, g, dL, dR, r.C);
    L.t_end("sgbm_cost");
    if (rc != L3D_OK) return rc;
    return sgbm_front_end(L, r);
}

// Left and right matcher of one frame (the right one sees the views swapped, camera/single_usb_stereo_camera.py:324-325):
// BT operands once per view, and -- when the pair of geometries is covered -- ONE pixel-cost pass that feeds both
// cost volumes (sgbm_cost_dual), else two single passes.
int sgbm_front_pair(Lane& L, const l3d_sgbm_params& pl, const l3d_sgbm_params& pr, const uint8_t* left,
                    const uint8_t* right, int W, int H, uint4* dL, uint4* dR, SgbmRun& rl, SgbmRun& rr) {
    int rc = sgbm_front_begin(L, pl, W, H, 0, rl);
    if (rc != L3D_OK) return rc;
    if ((rc = sgbm_front_begin(L, pr, W, H, 1, rr)) != L3D_OK) return rc;
    L3D_ARG(L, rl.g.ftzero == rr.g.ftzero, "left/right matcher preFilterCap differ");
    if (rl.g.width1 <= 0 && rr.g.width1 <= 0) return L3D_OK;
    if ((rc = sgbm_prefilter(L, left, W, H, rl.g.ftzero, dL)) != L3D_OK) return rc;
    if ((rc = sgbm_prefilter(L, right, W, H, rl.g.ftzero, dR)) != L3D_OK) return rc;
    if (rl.g.width1 > 0 && rr.g.width1 > 0 && sgbm_cost_dual_ok(rl.g, rr.g)) {
        L.t_begin("sgbm_cost");
        rc = sgbm_cost_dual(L, rl.g, rr.g, dL, dR, rl.C, rr.C);
        L.t_end("sgbm_cost");
        if (rc != L3D_OK) return rc;
        if ((rc = sgbm_front_end(L, rl)) != L3D_OK) return rc;
        return sgbm_front_end(L, rr);
    }
    // two single passes; each volume's horizontal paths follow its cost pass (the tail of C is still in L2)
    SgbmRun* runs[2] = {&rl, &rr};
    for (int i = 0; i < 2; i++) {
        SgbmRun& r = *runs[i];
        if (r.g.width1 <= 0) continue;
        L.t_begin("sgbm_cost");
        rc = i == 0 ? sgbm_cost_single(L, r.g, dL, dR, r.C) : sgbm_cost_single(L, r.g, dR, dL, r.C);
        L.t_end("sgbm_cost");
        if (rc != L3D_OK) return rc;
        if ((rc = sgbm_front_end(L, r)) != L3D_OK) return rc;
    }
    return L3D_OK;
}

// can the previous-row paths of this run go through the cluster-fused kernel?
bool sgbm_vgroup_ok(const SgbmRun& r) {
    return r.g.width1 > 0 && r.g.mode <= 1 && vgroup_supported(r.g.width1, r.g.HV, r.g.D);
}

// the previous-row paths with the direction-split scan kernels (any geometry and mode); the last path fuses
// the WTA unless the caller needs the finished S volume
int sgbm_middle_split(Lane& L, SgbmRun& r, bool keep_S) {
    const Geom& g = r.g;
    if (g.width1 <= 0) return L3D_OK;
    ScanArgs sa;
    scan_args_of(r, sa);
    int kinds[6], nk = 0;
    kinds[nk++] = 2;  // down: all modes
    if (g.mode <= 1) { kinds[nk++] = 3; kinds[nk++] = 4; }
    if (g.mode == 1) { kinds[nk++] = 5; kinds[nk++] = 6; kinds[nk++] = 7; }
    if (g.mode == 3) kinds[nk++] = 5;  // HH4: horizontal pair (front) + down + up
    // SGBM_3WAY keeps the stand-alone lean WTA: fused into the last scan it was slower (834 -> 696 frames/s at 1280x720:
    // the arg-min ballots sit on the scan's serial chain)
    const bool fuse_wta = !keep_S && g.mode != 2;
    for (int i = 0; i < nk; i++) {
        const int k = kinds[i];
        sa.kind = k; sa.store = 0;
        const int smode = (fuse_wta && i == nk - 1) ? SCAN_FINAL : SCAN_ACCUM;
        sa.lines_per_seg = (k == 2 || k == 5) ? g.width1 : g.width1 + g.H - 1;  // diagonals only with nseg == 1
        const int lines = g.nseg * sa.lines_per_seg;
        static const char* kind_names[8] = {"sgbm_scan_k0", "sgbm_scan_k1", "sgbm_scan_k2", "sgbm_scan_k3",
                                            "sgbm_scan_k4", "sgbm_scan_k5", "sgbm_scan_k6", "sgbm_scan_k7"};
        L.t_begin(kind_names[k]);
        int rc = launch_scan_np(L, g.NP, smode, sa, lines);
        L.t_end(kind_names[k]);
        if (rc != L3D_OK) return rc;
    }
    r.wta_done = fuse_wta;
    return L3D_OK;
}

// WTA (unless the last path did it), LR check, medianBlur(3), filterSpeckles -> disp
int sgbm_back(Lane& L, SgbmRun& r, int16_t* disp, SgbmDebug* dbg) {
    const Geom& g = r.g;
    const int W = r.W, H = r.H;
    const size_t npix = (size_t)W * H;
    const int16_t INVALID = (int16_t)((g.minD - 1) * 16);
    if (g.width1 > 0) {
        WtaArgs wa;
        wa.S = r.S; wa.raw = r.raw; wa.disp2key = r.d2; wa.W = W; wa.width1 = g.width1; wa.D = g.D; wa.nact = g.nact;
        wa.DPL = g.DPL; wa.minD = g.minD; wa.minX1 = g.minX1; wa.uniq = g.uniq;
        wa.HV = g.HV; wa.nseg = g.nseg;
        for (int s = 0; s < MAXSEG; s++) {
            wa.seg_vr0[s] = g.seg_vr0[s]; wa.seg_y0[s] = g.seg_y0[s] - g.seg_shift[s]; wa.seg_rows[s] = g.seg_rows[s]; wa.seg_emit[s] = g.seg_emit[s];
        }
        if (!r.wta_done) {  // (fused into the last aggregation pass otherwise: nothing to time here)
            L.t_begin("sgbm_wta");
            const int wgrid = cdiv(cdiv((long)g.HV * g.width1, 32), WTA_WARPS);
            if (g.mode != 2) {
                const bool full = g.nact == 32;
#define L3D_WTA(NPV)                                                                                         \
    do {                                                                                                     \
        if (full) L3D_LAUNCH(L, (sgbm_wta_lean_kernel<NPV, true>), wgrid, WTA_WARPS * 32, 0, wa);            \
        else L3D_LAUNCH(L, (sgbm_wta_lean_kernel<NPV, false>), wgrid, WTA_WARPS * 32, 0, wa);                \
    } while (0)
                if (g.NP == 1) L3D_WTA(1); else if (g.NP == 2) L3D_WTA(2); else if (g.NP == 4) L3D_WTA(4); else L3D_WTA(8);
#undef L3D_WTA
            } else {
                if (g.NP == 1) L3D_LAUNCH(L, sgbm_wta_lean3_kernel<1>, wgrid, WTA_WARPS * 32, 0, wa);
                else if (g.NP == 2) L3D_LAUNCH(L, sgbm_wta_lean3_kernel<2>, wgrid, WTA_WARPS * 32, 0, wa);
                else if (g.NP == 4) L3D_LAUNCH(L, sgbm_wta_lean3_kernel<4>, wgrid, WTA_WARPS * 32, 0, wa);
                else L3D_LAUNCH(L, sgbm_wta_lean3_kernel<8>, wgrid, WTA_WARPS * 32, 0, wa);
            }
            L.t_end("sgbm_wta");
        }
        L3D_LAUNCH(L, sgbm_lrcheck_kernel, dim3(cdiv(g.width1, 128), H), 128, 0, r.raw, r.d2, W, H, g.minX1, g.maxX1, g.minD, g.d12);
        if (dbg) {
            const size_t nvol = (size_t)g.HV * g.width1 * g.D;
            if (dbg->C) L3D_CHECK(L, cudaMemcpyAsync(dbg->C, r.C, nvol * 2, cudaMemcpyDeviceToDevice, L.stream));
            if (dbg->S) L3D_CHECK(L, cudaMemcpyAsync(dbg->S, r.S, nvol * 2, cudaMemcpyDeviceToDevice, L.stream));
        }
    }
    if (dbg && dbg->raw) L3D_CHECK(L, cudaMemcpyAsync(dbg->raw, r.raw, npix * 2, cudaMemcpyDeviceToDevice, L.stream));
    // --- medianBlur(3) then filterSpeckles, as StereoSGBM::compute does
    int rc = dev_median3(L, r.raw, W, H, disp);
    if (rc != L3D_OK) return rc;
    if (r.p.speckleWindowSize > 0) rc = dev_speckles(L, disp, W, H, INVALID, r.p.speckleWindowSize, 16 * r.p.speckleRange);
    return rc;
}

// the cluster-fused middle of a set of runs that share one geometry (one launch per pass); the last pass
// also does the WTA unless the caller needs the finished S volumes
int sgbm_middle_vgroup(Lane& L, SgbmRun* const* runs, int nruns, bool keep_S) {
    if (nruns <= 0) return L3D_OK;
    const Geom& g = runs[0]->g;
    std::vector<const int16_t*> Cp(nruns);
    std::vector<int16_t*> Sp(nruns);
    std::vector<VGroupWta> wta(nruns);
    for (int i = 0; i < nruns; i++) {
        const Geom& h = runs[i]->g;
        L3D_ARG(L, h.width1 == g.width1 && h.HV == g.HV && h.D == g.D && h.P1 == g.P1 && h.P2 == g.P2 && h.mode == g.mode &&
                       runs[i]->W == runs[0]->W,
                "vgroup: runs of one launch must share geometry and penalties");
        Cp[i] = runs[i]->C; Sp[i] = runs[i]->S;
        wta[i] = VGroupWta{runs[i]->raw, runs[i]->d2, runs[i]->W, h.minD, h.minX1, h.uniq};
        runs[i]->wta_done = !keep_S;
    }
    const VGroupWta* last = keep_S ? nullptr : wta.data();
    L.t_begin("sgbm_vgroup_down");
    int rc = dev_sgbm_vgroup(L, Cp.data(), Sp.data(), nruns, g.width1, g.HV, g.D, g.P1, g.P2, +1, g.mode == 1 ? nullptr : last);
    L.t_end("sgbm_vgroup_down");
    if (rc != L3D_OK) return rc;
    if (g.mode == 1) {
        L.t_begin("sgbm_vgroup_up");
        rc = dev_sgbm_vgroup(L, Cp.data(), Sp.data(), nruns, g.width1, g.HV, g.D, g.P1, g.P2, -1, last);
        L.t_end("sgbm_vgroup_up");
    }
    return rc;
}

// can all eight paths of this geometry go through the wavefront kernel?  (MODE_HH only: its two passes carry four paths each)
// L3D_VWAVE (read at every call; the frame pipeline calls this once, when it is created, so that a test can switch it
// per pipeline): 0 = never, 1 = wherever the kernel covers the geometry,
// unset = where it is the faster choice (vwave_pays)
bool sgbm_vwave_ok(int width1, int H, int D, int mode) {
    const char* e = getenv("L3D_VWAVE");
    const int policy = e ? atoi(e) : -1;
    if (policy == 0 || mode != 1 || width1 <= 0) return false;
    return policy == 1 ? vwave_supported(width1, H, D) : vwave_pays(width1, H, D);
}

// MODE_HH's eight paths of a set of runs that share one geometry: pass 1 (left-to-right, down-right, down, down-left)
// writes S, pass 2 (the mirrored four) accumulates and runs the winner-takes-all on the finished rows.
int sgbm_middle_vwave(Lane& L, SgbmRun* const* runs, int nruns) {
    if (nruns <= 0) return L3D_OK;
    const Geom& g = runs[0]->g;
    std::vector<const int16_t*> Cp(nruns);
    std::vector<int16_t*> Sp(nruns);
    std::vector<VGroupWta> wta(nruns);
    for (int i = 0; i < nruns; i++) {
        const Geom& h = runs[i]->g;
        L3D_ARG(L, h.width1 == g.width1 && h.HV == g.HV && h.D == g.D && h.P1 == g.P1 && h.P2 == g.P2 && h.mode == 1 &&
                       runs[i]->W == runs[0]->W && runs[i]->no_hpair,
                "vwave: runs of one launch must share geometry and penalties");
        Cp[i] = runs[i]->C; Sp[i] = runs[i]->S;
        wta[i] = VGroupWta{runs[i]->raw, runs[i]->d2, runs[i]->W, h.minD, h.minX1, h.uniq, runs[i]->wrec};
        runs[i]->wta_done = true;
    }
    L.t_begin("sgbm_vwave_down");
    int rc = dev_sgbm_vwave(L, Cp.data(), Sp.data(), nruns, g.width1, g.HV, g.D, g.P1, g.P2, +1, nullptr);
    L.t_end("sgbm_vwave_down");
    if (rc != L3D_OK) return rc;
    L.t_begin("sgbm_vwave_up");
    rc = dev_sgbm_vwave(L, Cp.data(), Sp.data(), nruns, g.width1, g.HV, g.D, g.P1, g.P2, -1, wta.data());
    L.t_end("sgbm_vwave_up");
    return rc;
}

int dev_sgbm(Lane& L, const l3d_sgbm_params& p, const uint8_t* left, const uint8_t* right, int W, int H,
             int16_t* disp, SgbmDebug* dbg) {
    const size_t npix = (size_t)W * H;
    uint4* dL = L.get<uint4>(S_DESC_L, 2 * npix);  // two operand planes per view (sgbm_prefilter_kernel)
    uint4* dR = L.get<uint4>(S_DESC_R, 2 * npix);
    SgbmRun r;
    int rc = sgbm_front(L, p, left, right, W, H, 0, dL, dR, true, r);
    if (rc != L3D_OK) return rc;
    // L3D_VGROUP=1 forces the cluster-fused kernel even for a single run (tests); by default a lone run uses
    // the direction-split kernels, which spread one volume over all SMs
    static const bool force_vgroup = getenv("L3D_VGROUP") && atoi(getenv("L3D_VGROUP")) > 0;
    if (force_vgroup && sgbm_vgroup_ok(r)) {
        SgbmRun* one[1] = {&r};
        rc = sgbm_middle_vgroup(L, one, 1, dbg && dbg->S);
    } else {
        rc = sgbm_middle_split(L, r, dbg && dbg->S);
    }
    if (rc != L3D_OK) return rc;
    return sgbm_back(L, r, disp, dbg);
}

}  // namespace l3d
