// sgbm_cost.cu -- BT operand planes and cost volumes of cv2.StereoSGBM (SURVEY A3), bit-exact.
//
// Replaces the pixel-cost / block-sum stage of stereo_matcher.compute / right_matcher.compute of the reference
// (camera/single_usb_stereo_camera.py:252-274 parameters, :324-325 calls).
//
// Kernels:
//   sgbm_prefilter_kernel     x-Sobel clip + half-pixel min/max, as pixel-pair operand entries (2 planes x 16 B / pixel)
//   sgbm_cost_dual_kernel     Birchfield-Tomasi pixel cost -> blockSize^2 box sum -> C (+P2) of one or both matchers of a
//                             frame at block 5 / D 64, block 9 / D 128, block 11 / D 256 (one volume: single-segment, or
//                             SGBM_3WAY's striped at block 5 / D 64 and block 9 / D 128; both: single-segment)
//   sgbm_cost_kernel          the block-synchronous form: every other geometry, SGBM_3WAY's at block 11 / D 256 among them
#include <map>
#include <mutex>

#include "sgbm.cuh"

namespace l3d {

constexpr int MAXBAND = 64;
// One band of a cost pass: volume rows vr0 .. vr0 + rows - 1 from image rows y0 .. y0 + rows - 1.  The vertical window
// clamps to image rows clo .. H - 1, so the box sum restarts at the top of the band's segment (SGBM_3WAY stripe, else
// the image).
struct CostBand {
    int vr0, y0, rows, clo;
};
// ------------------------------------------------------------------------------------------
// prefilter: per pixel and channel (0 = clipped x-Sobel, 1 = intensity) the Birchfield-Tomasi
// operands as signed 16-bit values, ready for packed s16x2 DPX arithmetic:
//   desc.x = v | (-v) << 16,  desc.y = lo | (-hi) << 16   (channel 0)      desc.z, desc.w (channel 1)
// where lo / hi = min / max of v and its two half-pixel interpolants.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void pre_pixel(const uint8_t* __restrict__ img, int W, int H, int y, int x,
                                          int ftzero, int& c0, int& c1) {
    if (x <= 0 || x >= W - 1) { c0 = ftzero; c1 = ftzero; return; }
    const uint8_t* r = img + (size_t)y * W;
    const uint8_t* rn = img + (size_t)(y > 0 ? y - 1 : y) * W;
    const uint8_t* rs = img + (size_t)(y < H - 1 ? y + 1 : y) * W;
    int g = ((int)r[x + 1] - (int)r[x - 1]) * 2 + (int)rn[x + 1] - (int)rn[x - 1] + (int)rs[x + 1] - (int)rs[x - 1];
    c0 = min(max(g, -ftzero), ftzero) + ftzero;
    c1 = r[x];
}

__device__ __forceinline__ uint32_t pack_s16(int lo, int hi) { return ((uint32_t)lo & 0xffffu) | ((uint32_t)hi << 16); }

// Output: two planes of W*H uint4 (plane c = channel c).  Entry x of a row holds the operands of the pixel PAIR
// (x+1, x) -- low halves pixel x+1, high halves pixel x -- exactly the layout the cost kernel's packed
// arithmetic wants for the disparity pair (d, d+1) of a left pixel (x - d = x_pair + 1):
//   .x = v | v' << 16,  .y = -v | -v' << 16,  .z = lo | lo' << 16,  .w = -hi | -hi' << 16     (' = pixel x)
// so a CTA's per-row operand table is a contiguous run of entries that one bulk async copy (TMA) moves
// into shared memory with no register staging; the left pixel's own operands are the high halves.
constexpr int PRE_THREADS = 128;
__global__ void __launch_bounds__(PRE_THREADS) sgbm_prefilter_kernel(const uint8_t* __restrict__ img, int W, int H,
                                                                     int ftzero, uint4* __restrict__ desc) {
    __shared__ int sv[6][PRE_THREADS + 1];
    const int t = threadIdx.x;
    const int x0 = blockIdx.x * PRE_THREADS, y = blockIdx.y;
    auto vals = [&](int x, int slot) {
        int a0, a1, b0, b1, c0, c1;
        pre_pixel(img, W, H, y, x, ftzero, b0, b1);
        int lo0 = b0, hi0 = b0, lo1 = b1, hi1 = b1;
        if (x > 0) {
            pre_pixel(img, W, H, y, x - 1, ftzero, a0, a1);
            int t0 = (b0 + a0) >> 1, t1 = (b1 + a1) >> 1;
            lo0 = min(lo0, t0); hi0 = max(hi0, t0); lo1 = min(lo1, t1); hi1 = max(hi1, t1);
        }
        if (x < W - 1) {
            pre_pixel(img, W, H, y, x + 1, ftzero, c0, c1);
            int t0 = (b0 + c0) >> 1, t1 = (b1 + c1) >> 1;
            lo0 = min(lo0, t0); hi0 = max(hi0, t0); lo1 = min(lo1, t1); hi1 = max(hi1, t1);
        }
        sv[0][slot] = b0; sv[1][slot] = lo0; sv[2][slot] = hi0; sv[3][slot] = b1; sv[4][slot] = lo1; sv[5][slot] = hi1;
    };
    vals(min(x0 + t, W - 1), t);
    if (t == PRE_THREADS - 1) vals(min(x0 + PRE_THREADS, W - 1), PRE_THREADS);  // pixel right of the block (clamped: pad)
    __syncthreads();
    const int x = x0 + t;
    if (x >= W) return;
    const size_t i = (size_t)y * W + x, plane = (size_t)W * H;
    desc[i] = make_uint4(pack_s16(sv[0][t + 1], sv[0][t]), pack_s16(-sv[0][t + 1], -sv[0][t]),
                         pack_s16(sv[1][t + 1], sv[1][t]), pack_s16(-sv[2][t + 1], -sv[2][t]));
    desc[plane + i] = make_uint4(pack_s16(sv[3][t + 1], sv[3][t]), pack_s16(-sv[3][t + 1], -sv[3][t]),
                                 pack_s16(sv[4][t + 1], sv[4][t]), pack_s16(-sv[5][t + 1], -sv[5][t]));
}

// ------------------------------------------------------------------------------------------
// cost volume: C[y][x][d] = P2 + sum over the blockSize^2 window of the BT pixel cost
// ------------------------------------------------------------------------------------------
// A CTA owns TX output columns (TXH = TX + 2*SW2 computed columns) of a band of rows and walks the
// band top to bottom.  Per image row:
//   tables  thread 0 issues two bulk async copies (cp.async.bulk, mbarrier completion) that bring the row's
//           right-image operand entries (prefilter layout above) into shared memory TWO rows ahead
//   phase A thread <-> (column, every (256/TXH)-th disparity pair): BT cost of both channels in
//           10 VIADD/VIADDMNMX/VIMNMX.S16x2 ops per two disparities -> pd[dp][col] (row stride TXH+1);
//           the thread's left operands sit in registers (loaded one row ahead)
//   phase B thread <-> (disparity pair, group of columns): running horizontal box sum along its
//           columns, vertical running sum against a ring of the last blockSize row sums, C store
//           (a warp writes 128 contiguous bytes per column)
// pd is double-buffered, so ONE block barrier per row separates {phase A of row k+1, phase B of row k}
// from the next pair.  All sums are wrap-around u16 like OpenCV's int16 arithmetic.
struct CostArgs {
    const uint4* Ldesc; const uint4* Rdesc; int16_t* C;  // two planes each (channel 0, channel 1)
    int W, H, minD, D, minX1, width1, SW2, bs, P2, TX, TXH;
    int nxg, cpg;  // phase B: column groups per CTA, columns per group
    unsigned* flags;  // bit 0 is set when a cost value reaches 32768 (OpenCV's int16 would wrap there; see make_geom)
    int nbands;
    CostBand band[MAXBAND];
};

constexpr int COST_THREADS = 512;
constexpr int COST_MAXCPG = 8;

__device__ __forceinline__ uint32_t bt_pair(uint32_t U, uint32_t nU, uint32_t U0, uint32_t nU1, const uint4& r) {
    // r = (V, -V, V0, -V1) pairs; max(0, u - v1, v0 - u) and max(0, v - u1, u0 - v), then the smaller.
    // One VIADD.16x2 + one VIADDMNMX.S16x2.RELU per term: no zero operand to materialise.
    const uint32_t t = __viaddmax_s16x2_relu(r.z, nU, __vadd2(U, r.w));
    const uint32_t q = __viaddmax_s16x2_relu(r.y, U0, __vadd2(r.x, nU1));
    return __vmins2(t, q);
}

__device__ __forceinline__ void cost_mbar_init(uint32_t bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void cost_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cost_mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "COST_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra COST_DONE_%=;\n\t"
        "bra COST_WAIT_%=;\n\t"
        "COST_DONE_%=:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void cost_bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

// NIT: phase A items (disparity pairs) per thread and row when known at compile time (D/2 / (512/TXH)), 0 = generic
// BS:  blockSize when known at compile time (phase B then keeps its window in registers), 0 = generic
// DD:  numDisparities, TXHT: tile width incl. halo when known at compile time (all strides become immediates), 0 = generic
template <int NIT, int BS, int DD, int TXHT>
__global__ void __launch_bounds__(COST_THREADS, 1) sgbm_cost_kernel(const CostArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int bs = BS ? BS : a.bs, SW2 = BS ? BS / 2 : a.SW2, D = DD ? DD : a.D, D2 = D >> 1;
    const int TXH = TXHT ? TXHT : a.TXH, TX = TXH - 2 * SW2;
    const int width1 = a.width1, W = a.W;
    const int tid = threadIdx.x;
    const int b = blockIdx.y, x0 = blockIdx.x * TX;
    const int y0 = a.band[b].y0, rows = a.band[b].rows, clo = a.band[b].clo, chi = a.H - 1, vr0 = a.band[b].vr0;
    const int xa = min(max(x0 - SW2, 0), width1 - 1);
    const int xb = min(max(x0 + TXH - 1 - SW2, 0), width1 - 1);
    const int xr_base = xa + a.minX1 - (a.minD + D - 1);  // lowest right pixel any pair reads
    const int nE = (xb - xa) + D - 1;                      // right operand entries (pair = pixels e+1, e)
    const int PS = TXH + 1;                                // pd row stride (bank-conflict-free both ways)
    const size_t plane = (size_t)W * a.H;
    // smem carve-up: operand tables [2 stages][R0 | R1][nEmax], pixel costs [2][D2][PS], ring [bs][TX][D2], 2 mbarriers
    const int nEmax = TXH + D;
    const int tab_u4 = 2 * nEmax;                          // uint4 per operand table stage
    uint4* tabs = (uint4*)smem_raw;
    uint32_t* pdb = (uint32_t*)(tabs + 2 * tab_u4);
    uint32_t* ring = pdb + 2 * D2 * PS;
    const uint32_t bars = (uint32_t)__cvta_generic_to_shared(ring + (size_t)bs * TX * D2);
    // phase A role
    const int ca = tid % TXH, dpa0 = tid / TXH, dpa_step = COST_THREADS / TXH;
    const int xca = min(max(x0 - SW2 + ca, 0), width1 - 1);
    // phase B role
    const int dpb = tid % D2, xg = tid / D2;
    const int cb0 = xg * a.cpg;                            // first output column (tile coordinates)
    const int ncb = xg < a.nxg ? max(0, min(min(a.cpg, TX - cb0), width1 - (x0 + cb0))) : 0;
    const uint32_t p2x2 = (uint32_t)a.P2 * 0x10001u;
    uint32_t crun[COST_MAXCPG];
#pragma unroll
    for (int j = 0; j < COST_MAXCPG; j++) crun[j] = p2x2;
    uint32_t ovf = 0;
    const int nk = rows + bs - 1;
    const int nitA = NIT ? NIT : (dpa0 < D2 ? (D2 - dpa0 + dpa_step - 1) / dpa_step : 0);  // phase A items of this thread

    auto row_of = [&](int k) { return min(max(y0 - SW2 + k, clo), chi); };
    auto issue_tables = [&](int k) {  // thread 0: both channels' operand entries of band row k -> stage k & 1
        const uint32_t bar = bars + 8 * (k & 1);
        const uint32_t bytes = (uint32_t)nE * 16u;
        const uint4* src = a.Rdesc + (size_t)row_of(k) * W + xr_base;
        uint4* dst = tabs + (k & 1) * tab_u4;
        cost_mbar_expect_tx(bar, 2 * bytes);
        cost_bulk_g2s((uint32_t)__cvta_generic_to_shared(dst), src, bytes, bar);
        cost_bulk_g2s((uint32_t)__cvta_generic_to_shared(dst + nEmax), src + plane, bytes, bar);
    };
    if (tid == 0) {
        cost_mbar_init(bars, 1);
        cost_mbar_init(bars + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        issue_tables(0);
        if (nk > 1) issue_tables(1);
    }
    // left operands of this thread's column: entry of pixel xca + minX1, loaded one row ahead
    const uint4* Lcol = a.Ldesc + xca + a.minX1;
    uint4 l0 = Lcol[(size_t)row_of(0) * W], l1 = Lcol[plane + (size_t)row_of(0) * W];
    __syncthreads();  // mbarrier init visible to every waiter

    auto phase_a = [&](int k) {  // pixel costs of band row k into pd[k & 1]
        // broadcast the left pixel's operands (high halves of its entry) to both halves
        const uint32_t u0 = __byte_perm(l0.x, l0.x, 0x3232), nu0 = __byte_perm(l0.y, l0.y, 0x3232);
        const uint32_t ul0 = __byte_perm(l0.z, l0.z, 0x3232), nuh0 = __byte_perm(l0.w, l0.w, 0x3232);
        const uint32_t u1 = __byte_perm(l1.x, l1.x, 0x3232), nu1 = __byte_perm(l1.y, l1.y, 0x3232);
        const uint32_t ul1 = __byte_perm(l1.z, l1.z, 0x3232), nuh1 = __byte_perm(l1.w, l1.w, 0x3232);
        if (k + 1 < nk) {  // next row's left operands: in flight during this row's arithmetic
            const size_t ro = (size_t)row_of(k + 1) * W;
            l0 = Lcol[ro]; l1 = Lcol[plane + ro];
        }
        cost_mbar_wait(bars + 8 * (k & 1), (uint32_t)((k >> 1) & 1));
        // this thread's disparity pairs dpa0, dpa0 + dpa_step, ...: table entry and pd slot move by constant strides
        const uint4* r0p = tabs + (k & 1) * tab_u4 + (xca - xa + D - 2 - 2 * dpa0);
        const uint4* r1p = r0p + nEmax;
        uint32_t* pdp = pdb + (k & 1) * D2 * PS + dpa0 * PS + ca;
        const int rstep = 2 * dpa_step, pstep = dpa_step * PS;
        if (NIT) {
            // batches of 4 items: all table loads first (the compiler cannot hoist them over the pd stores itself,
            // both are shared-memory accesses), then the arithmetic, then the stores
            constexpr int NB = 4;
#pragma unroll
            for (int i0 = 0; i0 < (NIT ? NIT : 1); i0 += NB) {
                uint4 e0[NB], e1[NB];
#pragma unroll
                for (int i = 0; i < NB; i++) { e0[i] = r0p[-(i0 + i) * rstep]; e1[i] = r1p[-(i0 + i) * rstep]; }
                uint32_t c[NB];
#pragma unroll
                for (int i = 0; i < NB; i++) {
                    const uint32_t c0 = bt_pair(u0, nu0, ul0, nuh0, e0[i]);
                    const uint32_t c1 = bt_pair(u1, nu1, ul1, nuh1, e1[i]);
                    c[i] = c0 + ((c1 >> 2) & 0x3fff3fffu);
                }
#pragma unroll
                for (int i = 0; i < NB; i++) pdp[(i0 + i) * pstep] = c[i];
            }
        } else {
#pragma unroll 4
            for (int i = 0; i < nitA; i++) {
                const uint32_t c0 = bt_pair(u0, nu0, ul0, nuh0, *r0p);
                const uint32_t c1 = bt_pair(u1, nu1, ul1, nuh1, *r1p);
                *pdp = c0 + ((c1 >> 2) & 0x3fff3fffu);
                r0p -= rstep; r1p -= rstep; pdp += pstep;
            }
        }
    };
    // Box sums.  Every packed half stays below 2^16 for the supported parameter range (checked on the
    // host), so plain 32-bit adds on the u16x2 pairs are exact: no carry crosses the halves.
    const uint32_t* ppb = pdb + dpb * PS + cb0;                 // + (k & 1) * D2 * PS per row
    uint32_t* rpb = ring + (size_t)cb0 * D2 + dpb;              // + slot * TX * D2 per row
    uint32_t* Cdst = (uint32_t*)(a.C + ((ptrdiff_t)(vr0 - (bs - 1)) * width1 + x0 + cb0) * D) + dpb;  // row k: + k * width1 * D2
    const size_t crow = (size_t)width1 * D2;
    int slot = 0;                                               // ring slot of row k (k % bs without the division)
    auto phase_b = [&](int k) {
        if (BS && ncb > 0) {
            // all shared-memory loads first (window taps, ring entries that drop out), then the sums, then the stores:
            // the compiler cannot move a load over the ring stores by itself
            const uint32_t* pp = ppb + (k & 1) * D2 * PS;       // pp[j + i]: output column cb0 + j, tap i
            uint32_t* rp = rpb + (size_t)slot * TX * D2;
            const bool sub = k >= bs, emit = k >= bs - 1;
            constexpr int NV = COST_MAXCPG + (BS ? BS : 1) - 1;
            uint32_t pv[NV], old[COST_MAXCPG], hs[COST_MAXCPG];
#pragma unroll
            for (int i = 0; i < NV; i++) pv[i] = pp[i];         // taps beyond this group's columns are never used
#pragma unroll
            for (int j = 0; j < COST_MAXCPG; j++) old[j] = (sub && j < ncb) ? rp[j * D2] : 0u;
            uint32_t h = 0;
#pragma unroll
            for (int i = 0; i < (BS ? BS : 1); i++) h += pv[i];
#pragma unroll
            for (int j = 0; j < COST_MAXCPG; j++) {
                if (j > 0) h = h + pv[j + (BS ? BS : 1) - 1] - pv[j - 1];
                hs[j] = h;
                crun[j] = crun[j] + h - old[j];
            }
#pragma unroll
            for (int j = 0; j < COST_MAXCPG; j++) {
                if (j < ncb) {
                    rp[j * D2] = hs[j];
                    ovf |= crun[j];
                    if (emit) Cdst[j * D2] = crun[j];
                }
            }
        } else if (ncb > 0) {
            const uint32_t* pp = ppb + (k & 1) * D2 * PS;       // pp[j + i]: output column cb0 + j, tap i
            uint32_t h = 0;
#pragma unroll 3
            for (int i = 0; i < bs; i++) h += pp[i];
            uint32_t* rp = rpb + (size_t)slot * TX * D2;
            const bool sub = k >= bs, emit = k >= bs - 1;
#pragma unroll
            for (int j = 0; j < COST_MAXCPG; j++) {
                if (j < ncb) {
                    if (j > 0) h = h + pp[j + bs - 1] - pp[j - 1];
                    uint32_t c = crun[j] + h;
                    if (sub) c -= rp[j * D2];
                    rp[j * D2] = h;
                    crun[j] = c;
                    ovf |= c;
                    if (emit) Cdst[j * D2] = c;
                }
            }
        }
        Cdst += crow;
        slot = slot + 1 == bs ? 0 : slot + 1;
    };
    phase_a(0);
    for (int k = 0; k < nk; k++) {
        __syncthreads();  // pd[k & 1] complete; stage k & 1 of the tables and pd[(k + 1) & 1] are free again
        if (tid == 0 && k + 2 < nk) issue_tables(k + 2);
        if (k + 1 < nk) phase_a(k + 1);
        phase_b(k);
    }
    if ((ovf & 0x80008000u) && a.flags) atomicOr(a.flags, 1u);
}

// ------------------------------------------------------------------------------------------
// cost volume of one matcher, or of BOTH matchers of a frame from one pixel-cost pass, with staged rows
// (block 5 / D 64, block 9 / D 128, block 11 / D 256)
// ------------------------------------------------------------------------------------------
// Same tile / band decomposition and the same arithmetic as sgbm_cost_kernel, but the disparity pairs are split over the
// 16 warps (DPW = D/32 pairs each) and BOTH phases of a pair stay in one warp: the warp computes the pixel costs of its
// pairs for all TXH tile columns (lane <-> columns lane + 32 h), writes them to a private strip of shared memory, and
// sums them itself (lane <-> pair x group of columns) against a private ring of row sums.  There is no block-wide
// barrier in the row loop: warps meet at the mbarriers of the operand-table ring (full: TMA bulk copies landed; empty:
// all 16 warps are done reading a stage) and of the staged rows below, so one warp's shared-memory latency is covered
// by another warp's arithmetic.  The left operands come in with the same bulk copies (contiguous run of the tile's
// columns; replicate-clamped tile edges index the run with a clamped column).  Each CTA walks one band of a band table
// (CostBand): a single-segment volume or the stripes of SGBM_3WAY, whose vertical windows restart at the stripe tops.
//
// The right matcher (minDisparity = -(D-1), views swapped: camera/single_usb_stereo_camera.py:277,325) evaluates the
// same Birchfield-Tomasi pixel costs as the left one -- the BT cost is symmetric in its two pixels -- and the box sum
// runs along x and y at a fixed disparity, so away from the replicate-clamped borders of the two width1 windows
//     C_right[y][x'][D-1-k] = C_left[y][x' + k - (D-1)][k]        (x, x' in width1 coordinates, k = 0 .. D-1)
// holds exactly, for x' in [SW2 + D-1, width1 - SW2) (derivation in DESIGN.md).  So:
//   role-0 CTAs  compute a tile of the LEFT matcher's volume, stage every finished row [column][disparity] in shared
//                memory, and all 16 warps then write the row out twice: as it is (coalesced 16-byte chunks, whole 256-byte
//                vectors) into C_left, and sheared into C_right for the columns RA <= x' < RB.  One right-volume word
//                (disparity indices 2w, 2w+1 of column x') is the high half of the staged word (column A = x' - 2w,
//                pair D/2-1-w) and the low half of the same pair one column to the left: two LDS + one PRMT.  The
//                words are walked along wrapped lines A = (s - 2w) mod TX so that consecutive lanes hold consecutive w
//                of the same x' (runs of ~TX/2 words = contiguous global bytes) and hit 32 different banks.  Tiles
//                step by TX - 1 columns: column A - 1 of a tile's first column belongs to the previous tile.
//   role-1 CTAs  compute, natively with the roles of the views exchanged, the right-volume columns the identity does
//                not cover (x' < RA: the first D-1+SW2 columns; x' >= RB: the last tile) -- about a sixth of a pass.
// Rows are handed from the phase-B lanes to the write-out by two shared-memory stages with full / empty mbarriers
// (split arrive / wait: a warp runs at most one row ahead of the slowest).
constexpr int CD_NS = 4;        // operand-table stages
constexpr int CD_PDS = 88;      // pixel-cost strip stride per pair
constexpr int CD_MAXT1 = 16;

struct DualArgs {
    const uint4* desc[2];       // BT operand planes of the left view [0] and the right view [1]
    int16_t* C[2];              // role r computes C[r]
    int W, H, width1, P2;
    int viewL[2], minD[2], minX1[2];  // role r: which view is its left image, its minDisparity, its minX1
    int ntiles[2], nbands[2];
    CostBand band[2][MAXBAND];  // role r: bands of every tile
    int stride0;                // role-0 tile origins: t * stride0; role-1 origins: x1[t]
    int x1[CD_MAXT1];
    int emit, RA, RB;           // role-0 tiles also write columns RA <= x' < RB of C[1]
    unsigned* flags;            // bit 0 is set when a cost value reaches 32768 (OpenCV's int16 would wrap there)
};

template <int BS, int DD>
struct CdCfg {
    // 64 computed columns per tile (two per lane in phase A) up to 128 disparities; 32 at 256 disparities, where the
    // ring of row sums (BS * D/2 * TX words) would not fit with more
    static constexpr int D = DD, D2 = DD / 2, SW2 = BS / 2, TXH = DD > 128 ? 32 : 64, NHH = TXH / 32, TX = TXH - 2 * SW2;
    static constexpr int NW = COST_THREADS / 32, DPW = D2 / NW, NG = 32 / DPW;
    // phase B: lane <-> (pair, group of CPG columns).  D = 256: 4 groups of 8 columns (the last one idle): with 6-column
    // groups no strip stride avoids 2-way bank conflicts on the tap loads
    static constexpr int CPG = DD > 128 ? 8 : (TX + NG - 1) / NG;
    static constexpr int PDS = DD > 128 ? 37 : CD_PDS;    // pixel-cost strip stride per pair (conflict-free tap loads)
    static constexpr int NEMAX = TXH + D;                 // right-operand entries per channel and stage
    static constexpr int STAGE_U4 = 2 * NEMAX + 2 * TXH;  // [R0 | R1 | L0 | L1]
    // staged row: column stride in words.  D = 128: 68 (== 4 mod 32: the phase-B lanes (pair, 7-column group) hit 32
    // banks, the sheared walk moves by -(2 * 68 + 1) == -9 words per lane and wraps by 56 * 68 == 0 mod 32); D = 256:
    // 129 (8-column groups: 8 * 129 == 8 mod 32); D = 64: 33 (2-way conflicts on the staging stores at best)
    static constexpr int CS = DD == 128 ? D2 + 4 : D2 + 1;
    static constexpr int NH = D2 / 32;                    // 32-word pieces of a right-volume vector
    static constexpr size_t smem_bytes() {
        return (size_t)CD_NS * STAGE_U4 * 16 + (size_t)D2 * PDS * 4 + (size_t)BS * D2 * TX * 4 + (size_t)2 * TX * CS * 4 +
               (size_t)(2 * CD_NS + 4) * 8 + 64;
    }
    static_assert(DPW >= 1 && 32 % DPW == 0 && CPG <= COST_MAXCPG && CPG * NG >= TX && D2 % 32 == 0, "tile geometry");
    static_assert(PDS >= ((TX - 1) / CPG) * CPG + CPG + BS - 1, "strip stride covers the last active group's taps");
};

__device__ __forceinline__ void cost_mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

template <int BS, int DD>
__global__ void __launch_bounds__(COST_THREADS, 1) sgbm_cost_dual_kernel(const DualArgs a) {
    typedef CdCfg<BS, DD> K;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int D = K::D, D2 = K::D2, SW2 = K::SW2, TXH = K::TXH, TX = K::TX;
    constexpr int NW = K::NW, DPW = K::DPW, CPG = K::CPG, NEMAX = K::NEMAX, STAGE_U4 = K::STAGE_U4, CS = K::CS, NH = K::NH;
    constexpr int NHH = K::NHH, PDS = K::PDS;
    const int width1 = a.width1, W = a.W;
    const int lane = threadIdx.x & 31;
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    // ---- CTA -> (role, tile, band)
    int cta = blockIdx.x;
    const int n0 = a.ntiles[0] * a.nbands[0];
    const int role = cta >= n0 ? 1 : 0;
    if (role) cta -= n0;
    const int nb = a.nbands[role];
    const int tile = cta / nb, b = cta - tile * nb;
    const int x0 = role ? a.x1[tile] : tile * a.stride0;
    const int y0 = a.band[role][b].y0, rows = a.band[role][b].rows, clo = a.band[role][b].clo, vr0 = a.band[role][b].vr0;
    const int chi = a.H - 1;
    const uint4* __restrict__ Ldesc = a.desc[a.viewL[role]];
    const uint4* __restrict__ Rdesc = a.desc[1 - a.viewL[role]];
    const int minD = a.minD[role], minX1 = a.minX1[role];
    const bool emitR = role == 0 && a.emit != 0;
    // columns of the own volume this tile writes (role 0 tiles overlap by one column when they feed the shear)
    const int next0 = role ? x0 + TX : x0 + a.stride0;
    const int ncopy = next0 < width1 ? min(TX, next0 - x0) : width1 - x0;

    const int xa = min(max(x0 - SW2, 0), width1 - 1);
    const int xb = min(max(x0 + TXH - 1 - SW2, 0), width1 - 1);
    const int xr_base = xa + minX1 - (minD + D - 1);
    const int nE = (xb - xa) + D - 1;
    const size_t plane = (size_t)W * a.H;
    const int lc0 = max(0, SW2 - x0), lc1 = min(TXH, width1 - (x0 - SW2));
    uint4* tabs = (uint4*)smem_raw;                                              // [CD_NS][STAGE_U4]
    uint32_t* u32base = (uint32_t*)(tabs + CD_NS * STAGE_U4);
    uint32_t* pdw = u32base + warp * DPW * PDS;                               // this warp's pixel-cost strip [DPW][PDS]
    uint32_t* ringw = u32base + D2 * PDS + (size_t)warp * BS * DPW * TX;      // this warp's row sums [BS][DPW][TX]
    uint32_t* Ls = u32base + D2 * PDS + (size_t)BS * D2 * TX;                 // staged rows [2][TX][CS]
    const uint32_t bars = (uint32_t)__cvta_generic_to_shared(Ls + 2 * TX * CS);
    // bars + 8 s: full[s]; + 8 (CD_NS + s): empty[s]; + 8 (2 CD_NS + s): row staged[s]; + 8 (2 CD_NS + 2 + s): row written out[s]
    const uint32_t bar_lsf = bars + 8 * (2 * CD_NS), bar_lse = bars + 8 * (2 * CD_NS + 2);
    const int nk = rows + BS - 1;
    auto row_of = [&](int k) { return min(max(y0 - SW2 + k, clo), chi); };
    auto issue_tables = [&](int k) {
        const int s = k % CD_NS;
        const uint32_t bar = bars + 8 * s;
        const uint32_t rbytes = (uint32_t)nE * 16u, lbytes = (uint32_t)(lc1 - lc0) * 16u;
        const size_t ro = (size_t)row_of(k) * W;
        const uint4* rsrc = Rdesc + ro + xr_base;
        const uint4* lsrc = Ldesc + ro + (x0 - SW2 + lc0) + minX1;
        uint4* dst = tabs + s * STAGE_U4;
        cost_mbar_expect_tx(bar, 2 * rbytes + 2 * lbytes);
        cost_bulk_g2s((uint32_t)__cvta_generic_to_shared(dst), rsrc, rbytes, bar);
        cost_bulk_g2s((uint32_t)__cvta_generic_to_shared(dst + NEMAX), rsrc + plane, rbytes, bar);
        cost_bulk_g2s((uint32_t)__cvta_generic_to_shared(dst + 2 * NEMAX + lc0), lsrc, lbytes, bar);
        cost_bulk_g2s((uint32_t)__cvta_generic_to_shared(dst + 2 * NEMAX + TXH + lc0), lsrc + plane, lbytes, bar);
    };
    if (threadIdx.x == 0) {
        for (int s = 0; s < CD_NS; s++) { cost_mbar_init(bars + 8 * s, 1); cost_mbar_init(bars + 8 * (CD_NS + s), NW); }
        for (int s = 0; s < 2; s++) { cost_mbar_init(bar_lsf + 8 * s, NW); cost_mbar_init(bar_lse + 8 * s, NW); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        for (int k = 0; k < CD_NS - 1 && k < nk; k++) issue_tables(k);
    }
    __syncthreads();  // barrier init visible; the only block-wide barrier of the kernel

    // phase A role: tile columns lane and lane + 32, pairs dp0 .. dp0 + DPW - 1
    const int dp0 = warp * DPW;
    int eoff[NHH], lcol[NHH];
#pragma unroll
    for (int hh = 0; hh < NHH; hh++) {
        const int c = lane + 32 * hh;
        const int xc = min(max(x0 - SW2 + c, 0), width1 - 1);
        eoff[hh] = xc - xa + D - 2 - 2 * dp0;
        lcol[hh] = min(max(c, lc0), lc1 - 1);
    }
    // phase B role
    const int dpi = lane % DPW, g = lane / DPW;
    const int cb0 = g * CPG;
    const int ncb = max(0, min(min(CPG, TX - cb0), width1 - (x0 + cb0)));
    const uint32_t p2x2 = (uint32_t)a.P2 * 0x10001u;
    uint32_t crun[CPG];
#pragma unroll
    for (int j = 0; j < CPG; j++) crun[j] = p2x2;
    const uint32_t* ppb = pdw + dpi * PDS + cb0;
    uint32_t* rpb = ringw + dpi * TX + cb0;
    uint32_t* lsb = Ls + cb0 * CS + dp0 + dpi;                 // + stage * TX * CS, + j * CS
    int slot = 0;
    uint32_t ovf = 0;
    // write-out role: sheared walk constants, cw[h] = (-2 w) mod TX for w = 32 h + lane
    const int cw0 = (TX * 16 - 2 * lane) % TX;                 // + TX - (64 h) % TX per piece h
    uint32_t* Cown32 = (uint32_t*)a.C[role];
    uint32_t* Cother32 = (uint32_t*)a.C[1];

    auto write_out = [&](int er) {  // emitted row er of the band (volume row vr0 + er), staged in Ls[er & 1]
        const uint32_t* ls = Ls + (er & 1) * TX * CS;
        const size_t rowbase = (size_t)(vr0 + er) * width1;
        if (CS % 4 == 0) {
            constexpr int CPC = D2 / 4;                    // 16-byte chunks per column
            for (int q = threadIdx.x; q < ncopy * CPC; q += COST_THREADS) {
                const int col = q / CPC, part = q - col * CPC;
                const uint4 v = *(const uint4*)(ls + col * CS + part * 4);
                *(uint4*)(Cown32 + (rowbase + x0 + col) * D2 + part * 4) = v;
            }
        } else {
            for (int q = threadIdx.x; q < ncopy * D2; q += COST_THREADS) {
                const int col = q / D2, part = q - col * D2;
                Cown32[(rowbase + x0 + col) * D2 + part] = ls[col * CS + part];
            }
        }
        if (emitR) {
            // units (wrapped line s, 32-word piece h) are dealt to the warps round robin: unit = warp + NW i, so a warp
            // keeps its piece h = warp % NH and its line advances by NW / NH per unit -- column, staged-row address and
            // global address all move by constants (with one conditional wrap)
            constexpr int SSTEP = NW / NH;                     // line step per unit
            constexpr int NU = (TX * NH + NW - 1) / NW;        // units per warp (the last one may not exist)
            const int h = warp % NH, w = 32 * h + lane;
            int sline = warp / NH;
            int u = (sline + cw0 + TX * 16 - 64 * h) % TX;
            const uint32_t* lsp = ls + u * CS + (D2 - 1 - w);                           // column u; column u + 1 is CS further
            uint32_t* gp = Cother32 + (rowbase + x0 + u + 1 + 2 * w) * D2 + w;
            int xq = x0 + u + 1 + 2 * w;                       // right-volume column of this word
#pragma unroll
            for (int i = 0; i < NU; i++) {
                if (sline < TX && u < TX - 1 && xq >= a.RA && xq < a.RB) *gp = __byte_perm(lsp[CS], lsp[0], 0x5432);
                sline += SSTEP; u += SSTEP; lsp += SSTEP * CS; gp += SSTEP * D2; xq += SSTEP;
                if (u >= TX) { u -= TX; lsp -= TX * CS; gp -= TX * D2; xq -= TX; }
            }
        }
    };

    for (int k = 0; k <= nk; k++) {  // iteration nk only writes out the last row
        const int e = k - (BS - 1);  // row this iteration emits
        if (k < nk) {
            const int s = k % CD_NS;
            if (warp == (k & (NW - 1)) && k + CD_NS - 1 < nk) {
                if (lane == 0) {
                    const int kk = k + CD_NS - 1, sk = kk % CD_NS;
                    if (k >= 1) cost_mbar_wait(bars + 8 * (CD_NS + sk), (uint32_t)(((k - 1) / CD_NS) & 1));
                    issue_tables(kk);
                }
                __syncwarp();
            }
            cost_mbar_wait(bars + 8 * s, (uint32_t)((k / CD_NS) & 1));
            const uint4* T0 = tabs + s * STAGE_U4;
            // ---- phase A
#pragma unroll
            for (int hh = 0; hh < NHH; hh++) {
                const uint4 l0 = T0[2 * NEMAX + lcol[hh]], l1 = T0[2 * NEMAX + TXH + lcol[hh]];
                const uint32_t u0 = __byte_perm(l0.x, l0.x, 0x3232), nu0 = __byte_perm(l0.y, l0.y, 0x3232);
                const uint32_t ul0 = __byte_perm(l0.z, l0.z, 0x3232), nuh0 = __byte_perm(l0.w, l0.w, 0x3232);
                const uint32_t u1 = __byte_perm(l1.x, l1.x, 0x3232), nu1 = __byte_perm(l1.y, l1.y, 0x3232);
                const uint32_t ul1 = __byte_perm(l1.z, l1.z, 0x3232), nuh1 = __byte_perm(l1.w, l1.w, 0x3232);
                constexpr int NB = DPW < 4 ? DPW : 4;  // pairs per batch: all table loads, then the arithmetic, then the stores
#pragma unroll
                for (int i0 = 0; i0 < DPW; i0 += NB) {
                    uint4 e0[NB], e1[NB];
#pragma unroll
                    for (int i = 0; i < NB; i++) { e0[i] = T0[eoff[hh] - 2 * (i0 + i)]; e1[i] = T0[NEMAX + eoff[hh] - 2 * (i0 + i)]; }
                    uint32_t c[NB];
#pragma unroll
                    for (int i = 0; i < NB; i++) {
                        const uint32_t c0 = bt_pair(u0, nu0, ul0, nuh0, e0[i]);
                        const uint32_t c1 = bt_pair(u1, nu1, ul1, nuh1, e1[i]);
                        c[i] = c0 + ((c1 >> 2) & 0x3fff3fffu);
                    }
#pragma unroll
                    for (int i = 0; i < NB; i++) pdw[(i0 + i) * PDS + lane + 32 * hh] = c[i];
                }
            }
            __syncwarp();
            if (lane == 0) cost_mbar_arrive(bars + 8 * (CD_NS + s));
            // ---- phase B
            const bool emit = e >= 0;
            if (e >= 2) cost_mbar_wait(bar_lse + 8 * (e & 1), (uint32_t)(((e >> 1) - 1) & 1));  // row e - 2 written out
            if (ncb > 0) {
                uint32_t* rp = rpb + (size_t)slot * DPW * TX;
                uint32_t* lp = lsb + (e & 1) * TX * CS;
                const bool sub = k >= BS;
                constexpr int NV = CPG + BS - 1;
                uint32_t pv[NV], old[CPG], hs[CPG];
#pragma unroll
                for (int i = 0; i < NV; i++) pv[i] = ppb[i];
#pragma unroll
                for (int j = 0; j < CPG; j++) old[j] = (sub && j < ncb) ? rp[j] : 0u;
                uint32_t h = 0;
#pragma unroll
                for (int i = 0; i < BS; i++) h += pv[i];
#pragma unroll
                for (int j = 0; j < CPG; j++) {
                    if (j > 0) h = h + pv[j + BS - 1] - pv[j - 1];
                    hs[j] = h;
                    crun[j] = crun[j] + h - old[j];
                }
#pragma unroll
                for (int j = 0; j < CPG; j++) {
                    if (j < ncb) {
                        rp[j] = hs[j];
                        ovf |= crun[j];
                        if (emit) lp[j * CS] = crun[j];
                    }
                }
            }
            __syncwarp();  // the strip is rewritten by the next row's phase A; this warp's part of the staged row is complete
            slot = slot + 1 == BS ? 0 : slot + 1;
            if (emit && lane == 0) cost_mbar_arrive(bar_lsf + 8 * (e & 1));
        }
        if (e >= 1) {  // write out the previous row while the other warps finish this one
            cost_mbar_wait(bar_lsf + 8 * ((e - 1) & 1), (uint32_t)(((e - 1) >> 1) & 1));
            write_out(e - 1);
            __syncwarp();
            if (lane == 0) cost_mbar_arrive(bar_lse + 8 * ((e - 1) & 1));
        }
    }
    if ((ovf & 0x80008000u) && a.flags) atomicOr(a.flags, 1u);
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
int sgbm_prefilter(Lane& L, const uint8_t* img, int W, int H, int ftzero, uint4* desc) {
    dim3 pg(cdiv(W, PRE_THREADS), H);
    L3D_LAUNCH(L, sgbm_prefilter_kernel, pg, PRE_THREADS, 0, img, W, H, ftzero, desc);
    return L3D_OK;
}

// Splits every segment of g (SGBM_3WAY stripe, else the image) into n bands of ceil(rows / n) rows,
// n = min(nmax, rows / (2 blockSize)) but at least 1.  Returns the number of bands.
static int cost_bands(const Geom& g, int nmax, CostBand* band) {
    int nb = 0;
    for (int s = 0; s < g.nseg; s++) {
        const int rows = g.seg_rows[s];
        const int br = cdiv(rows, std::max(1, std::min(nmax, rows / (2 * g.bs))));
        for (int r0 = 0; r0 < rows; r0 += br) band[nb++] = {g.seg_vr0[s] + r0, g.seg_y0[s] + r0, std::min(br, rows - r0), g.seg_y0[s]};
    }
    return nb;
}

// nmax of cost_bands for a grid close to one wave of CTAs (one CTA per SM: the row-sum ring takes most of the shared
// memory) over xtiles column tiles
static int cost_wave_bands(const Geom& g, int xtiles) {
    const int want = std::max(1, NUM_SMS / xtiles);
    return std::max(1, std::min(want / g.nseg, MAXBAND / g.nseg));
}

// Band split of a single-segment launch of the staged kernel: nt0 role-0 tiles and nt1 role-1 tiles, every CTA walks
// (band rows + bs - 1) rows; one CTA per SM.  Picks the bands per tile of both roles that minimise the finish time of
// a greedy assignment of the CTAs (in launch order: role 0 first) to the SMs.  The result depends on the arguments
// alone and is computed once per process.
static void cost_pick_bands(int H, int bs, int nt0, int nt1, int& b0_out, int& b1_out) {
    static std::mutex mu;
    static std::map<long long, std::pair<int, int>> cache;
    const long long key = ((long long)H << 40) | ((long long)bs << 32) | ((long long)nt0 << 8) | nt1;
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(key);
    if (it == cache.end()) {
        // with role-1 tiles (both matchers' volumes), a role-0 row costs about 1.35 role-1 rows: it also writes the
        // sheared copy
        const double w0 = nt1 ? 1.35 : 1.0, w1 = 1.0;
        const int maxb = std::max(1, std::min(MAXBAND, H / (2 * bs)));
        double bestt = 1e30;
        int b0b = 1, b1b = 1;
        std::vector<double> sm(NUM_SMS);
        for (int b0 = 1; b0 <= maxb; b0++) {
            for (int b1 = 1; b1 <= (nt1 ? maxb : 1); b1++) {
                const double t0 = w0 * (cdiv(H, b0) + bs - 1), t1 = w1 * (cdiv(H, b1) + bs - 1);
                std::fill(sm.begin(), sm.end(), 0.0);
                const int n0 = nt0 * b0, n1 = nt1 * b1;
                if (n0 + n1 > 4096) continue;
                // CTAs of equal length: fill round-robin onto the earliest-free SM
                for (int i = 0; i < n0 + n1; i++) {
                    int k = 0;
                    for (int q = 1; q < NUM_SMS; q++) if (sm[q] < sm[k]) k = q;
                    sm[k] += i < n0 ? t0 : t1;
                }
                double t = 0;
                for (double v : sm) t = std::max(t, v);
                // inside the frame pipeline other kernels fill idle SMs, so total work (halo rows of short bands) counts too
                t += 0.3 * (n0 * t0 + n1 * t1) / NUM_SMS + 1e-3 * (b0 + b1);
                if (t < bestt) { bestt = t; b0b = b0; b1b = b1; }
            }
        }
        it = cache.emplace(key, std::make_pair(b0b, b1b)).first;
    }
    b0_out = it->second.first; b1_out = it->second.second;
}

// the (blockSize, numDisparities) pairs the staged kernel is instantiated for
static bool cost_dual_cfg(int bs, int D) { return (bs == 9 && D == 128) || (bs == 5 && D == 64) || (bs == 11 && D == 256); }

template <int BS, int DD>
static int launch_cost_dual(Lane& L, const DualArgs& da) {
    typedef CdCfg<BS, DD> K;
    const int ncta = da.ntiles[0] * da.nbands[0] + da.ntiles[1] * da.nbands[1];
    L3D_CHECK(L, cudaFuncSetAttribute((sgbm_cost_dual_kernel<BS, DD>), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)K::smem_bytes()));
    L3D_LAUNCH(L, (sgbm_cost_dual_kernel<BS, DD>), ncta, COST_THREADS, K::smem_bytes(), da);
    return L3D_OK;
}
static int launch_cost_dual_any(Lane& L, int bs, int D, const DualArgs& da) {
    if (bs == 9 && D == 128) return launch_cost_dual<9, 128>(L, da);
    if (bs == 5 && D == 64) return launch_cost_dual<5, 64>(L, da);
    if (bs == 11 && D == 256) return launch_cost_dual<11, 256>(L, da);
    set_err(L.err, "sgbm_cost_dual: no instantiation for blockSize %d / numDisparities %d", bs, D);
    return L3D_ERR_UNSUPPORTED;
}

static int cost_dual_tx(int bs, int D) { return (D > 128 ? 32 : 64) - 2 * (bs / 2); }

int sgbm_cost_single(Lane& L, const Geom& g, const uint4* dL, const uint4* dR, int16_t* C) {
    // SGBM_3WAY's striped volumes at block 11 / D 256 stay on the block-synchronous kernel's specialisation below: the
    // staged kernel's cost pass is about 6 % slower there in the frame pipeline (tools/kernel_times.py, 1920x1080, one
    // B200 at 1000 W)
    if (cost_dual_cfg(g.bs, g.D) && (g.nseg == 1 || g.D != 256)) {
        // the staged kernel, role 0 only: nothing is emitted into a second volume
        DualArgs da = {};
        da.desc[0] = dL; da.desc[1] = dR; da.C[0] = C;
        da.W = g.W; da.H = g.H; da.width1 = g.width1; da.P2 = g.P2;
        da.viewL[0] = 0; da.minD[0] = g.minD; da.minX1[0] = g.minX1;
        const int TX = cost_dual_tx(g.bs, g.D);
        da.stride0 = TX; da.ntiles[0] = cdiv(g.width1, TX);
        int nb = cost_wave_bands(g, da.ntiles[0]), nb1;
        if (g.nseg == 1) cost_pick_bands(g.H, g.bs, da.ntiles[0], 0, nb, nb1);
        da.nbands[0] = cost_bands(g, nb, da.band[0]);
        da.flags = L.flags;
        return launch_cost_dual_any(L, g.bs, g.D, da);
    }
    CostArgs ca;
    ca.Ldesc = dL; ca.Rdesc = dR; ca.C = C;
    ca.W = g.W; ca.H = g.H; ca.minD = g.minD; ca.D = g.D; ca.minX1 = g.minX1; ca.width1 = g.width1;
    ca.SW2 = g.SW2; ca.bs = g.bs; ca.P2 = g.P2; ca.flags = L.flags;
    const int D2 = g.D / 2;
    auto cost_smem = [&](int txh) {
        int tx = txh - 2 * g.SW2;
        return (size_t)2 * 2 * (txh + g.D) * 16 + (size_t)2 * D2 * (txh + 1) * 4 + (size_t)g.bs * tx * D2 * 4 + 16;
    };
    ca.nxg = std::max(1, COST_THREADS / D2);
    int TXH = 64;
    while (TXH > 2 * g.SW2 + 1 &&
           (cost_smem(TXH) > 200 * 1024 || cdiv(TXH - 2 * g.SW2, ca.nxg) > COST_MAXCPG)) TXH /= 2;
    L3D_ARG(L, TXH > 2 * g.SW2 && COST_THREADS % TXH == 0 && cost_smem(TXH) <= 200 * 1024 &&
                   cdiv(TXH - 2 * g.SW2, ca.nxg) <= COST_MAXCPG,
            "sgbm: blockSize / numDisparities combination exceeds the cost kernel's shared-memory tile");
    ca.TXH = TXH; ca.TX = TXH - 2 * g.SW2;
    ca.cpg = cdiv(ca.TX, ca.nxg);
    const int xtiles = cdiv(g.width1, ca.TX);
    ca.nbands = cost_bands(g, cost_wave_bands(g, xtiles), ca.band);
    const int dpa_step = COST_THREADS / TXH;
    const int nit = (D2 % dpa_step == 0) ? D2 / dpa_step : 0;
#define COST_CASE(KERN)                                                                                          \
    {                                                                                                            \
        L3D_CHECK(L, cudaFuncSetAttribute(KERN, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));       \
        L3D_LAUNCH(L, KERN, dim3(xtiles, ca.nbands), COST_THREADS, cost_smem(TXH), ca);                          \
    }
    // specialised for SGBM_3WAY at the configuration of c4 (D 256 / block 11)
    if (nit == 8 && g.bs == 11 && g.D == 256 && TXH == 32) COST_CASE((sgbm_cost_kernel<8, 11, 256, 32>))
    else COST_CASE((sgbm_cost_kernel<0, 0, 0, 0>))
#undef COST_CASE
    return L3D_OK;
}

bool sgbm_cost_dual_ok(const Geom& gl, const Geom& gr) {
    return cost_dual_cfg(gl.bs, gl.D) && gr.bs == gl.bs && gr.D == gl.D && gl.minD == 0 && gr.minD == -(gl.D - 1) &&
           gl.P2 == gr.P2 && gl.ftzero == gr.ftzero && gl.nseg == 1 && gr.nseg == 1 && gl.W == gr.W && gl.H == gr.H &&
           gl.width1 == gr.width1 && gl.width1 > 0;
}

int sgbm_cost_dual(Lane& L, const Geom& gl, const Geom& gr, const uint4* dLv, const uint4* dRv, int16_t* Cl, int16_t* Cr) {
    L3D_ARG(L, sgbm_cost_dual_ok(gl, gr), "sgbm_cost_dual geometry");
    const int D = gl.D, SW2 = gl.SW2, W1 = gl.width1, H = gl.H;
    const int TX = cost_dual_tx(gl.bs, D);
    DualArgs da = {};
    da.desc[0] = dLv; da.desc[1] = dRv; da.C[0] = Cl; da.C[1] = Cr;
    da.W = gl.W; da.H = H; da.width1 = W1; da.P2 = gl.P2;
    da.viewL[0] = 0; da.minD[0] = gl.minD; da.minX1[0] = gl.minX1;
    da.viewL[1] = 1; da.minD[1] = gr.minD; da.minX1[1] = gr.minX1;
    // role 0: the left volume in tiles that step by TX - 1 columns
    da.stride0 = TX - 1;
    da.ntiles[0] = W1 <= TX ? 1 : cdiv(W1 - TX, da.stride0) + 1;
    // role 1: right-volume columns outside the identity's domain, natively
    const int nbl = cdiv(D - 1 + SW2, TX);
    da.RA = std::min(nbl * TX, W1);
    da.RB = std::max(da.RA, W1 - TX);
    da.emit = da.RB > da.RA;
    int nt1 = 0;
    for (int x = 0; x < da.RA && nt1 < CD_MAXT1; x += TX) da.x1[nt1++] = x;
    L3D_ARG(L, nt1 * TX >= da.RA, "sgbm_cost_dual: border tiles");
    if (da.RB < W1) {
        L3D_ARG(L, nt1 < CD_MAXT1, "sgbm_cost_dual: border tiles");
        da.x1[nt1++] = da.RB;
    }
    da.ntiles[1] = nt1; da.flags = L.flags;
    int b0, b1;
    cost_pick_bands(H, gl.bs, da.ntiles[0], nt1, b0, b1);
    da.nbands[0] = cost_bands(gl, b0, da.band[0]);
    da.nbands[1] = cost_bands(gr, b1, da.band[1]);
    if (getenv("L3D_DEBUG_CLUSTERS"))
        fprintf(stderr, "[l3d] cost dual: %d x %d + %d x %d CTAs, RA %d RB %d\n", da.ntiles[0], da.nbands[0], nt1, da.nbands[1], da.RA, da.RB);
    return launch_cost_dual_any(L, gl.bs, D, da);
}

}  // namespace l3d
