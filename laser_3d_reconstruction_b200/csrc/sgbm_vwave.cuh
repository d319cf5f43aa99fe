// sgbm_vwave.cuh -- FOUR SGM paths per pass on a thread-block cluster, as a warp-skewed wavefront: the whole aggregation of
// cv2.StereoSGBM MODE_HH (camera/single_usb_stereo_camera.py:324-325) in two passes that move exactly the algorithmic
// bytes (SURVEY 8d: every pass reads C once and reads-or-writes S once).
//
// S is a saturating sum of eight non-negative path costs, so the paths may be grouped into passes freely:
//   pass 1 (rows top-down, columns left-to-right):   H from (x-1, y),  A from (x-1, y-1),  V from (x, y-1),  B from (x+1, y-1)
//   pass 2 = the same kernel on the volume mirrored in x and y: from (x+1, y), (x+1, y+1), (x, y+1), (x-1, y+1)
// H needs the LEFT neighbour of the same row, B the RIGHT neighbour of the previous row.  In row lock-step (sgbm_vgroup.cu)
// the two cannot share a pass.  Here warp g (owner of CPW adjacent columns, all warps of the cluster numbered left to
// right) simply runs one row BEHIND warp g-1: it exports the B state of its FIRST column early in a row and imports its
// right neighbour's (one row back, produced at about the same time) just before its LAST column.  Nothing is in
// lock-step: every warp streams its own rows of C (and S) by TMA bulk copies with its own mbarriers and talks to its two
// neighbours only, through double-buffered slots with full / empty mbarriers -- plain shared memory inside a CTA,
// st.async + remote arrive between the CTAs of the cluster.  The price of the skew is (warps per cluster - 1) row-times of
// pipeline fill and drain per pass.
//
// What it replaces: sgbm_scan_hpair_kernel (both horizontal paths: 4.3 volume-passes of DRAM traffic, because a pixel's
// two horizontal costs meet half a row apart) and the two sgbm_vgroup_kernel passes (3 + 2 volume-passes).
#pragma once
#include <cooperative_groups.h>

#include <type_traits>

#include "common.cuh"
#include "sgm_step.cuh"

namespace l3d {
namespace cg = cooperative_groups;

constexpr int VW_MAXCPW = 9;      // D <= 128: 16 warps per CTA, 128 registers per thread
constexpr int VW_MAXCPW256 = 13;  // D = 256: 8 warps per CTA, 255 registers per thread
constexpr int VW_MAXJOBS = 64;
constexpr int VW_MAXREG = 128;

struct VWaveArgs {
    const int16_t* C[VW_MAXJOBS];
    int16_t* S[VW_MAXJOBS];
    int width1, H, D, P1, P2;
    int dir;       // +1: pass 1 (rows top-down, strips left-to-right); -1: pass 2 (the volume mirrored in x and y)
    int cluster;   // CTAs per cluster (= per job)
    int W;         // image width (WTA outputs)
    uint32_t zero; // 0, as a value the compiler cannot see (sgm_step.cuh)
    uint2* rec[VW_MAXJOBS];   // last pass: per-pixel winner records [H][width1] for vw_finish_kernel
    int uniq[VW_MAXJOBS];
};

// shared memory per warp: C rows [2][CPW * B], S rows [2][CPW * B], left-edge slots [2][2 * (B + 16)], right-edge slots
// [2][B + 16], 10 mbarriers
// D = 256: the neighbour slots are single-buffered and the last pass adds the horizontal path's costs into the S row in
// place (no row of its own), so that 8 warps x 4 row buffers of 13 x 512 bytes fit 227 KB
static inline int vwave_warps(int D) { return D > 128 ? 8 : 16; }
// distance of a warp's two stage blocks [C row | S row | 64 bytes of mbarriers | three neighbour slots] (see the kernel),
// a multiple of 128 bytes so that both blocks' rows are aligned alike for the bulk copies
__host__ __device__ constexpr uint32_t vwave_delta(uint32_t rowb, uint32_t slot) { return (2 * rowb + 64 + 3 * slot + 127u) & ~127u; }
static inline size_t vwave_warp_bytes(int D, int cpw, bool last) {
    const uint32_t B = (uint32_t)D * 2, row = (uint32_t)cpw * B, slot = B + 16, delta = vwave_delta(row, slot);
    if (D > 128) return ((size_t)delta + 2 * row + 64 + 127) & ~(size_t)127;   // single-buffered slots: block 1 is [C | S | barriers]
    return 2 * (size_t)delta + (last ? row : 0);   // (rows are multiples of 128 bytes)
}
static inline size_t vwave_smem_bytes(int D, int cpw, bool last) { return vwave_warps(D) * vwave_warp_bytes(D, cpw, last) + 128; }

__device__ __forceinline__ void vw_mbar_init(uint32_t bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void vw_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void vw_mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// A barrier in another CTA of the cluster.  Only "slot free" signals travel this way: the consumer has READ the slot (its
// LDS results are in registers, the warp has re-converged) and nothing it wrote has to become visible to the producer, so
// the arrive is relaxed.  The release form costs MEMBAR.ALL.GPU + ERRBAR + CGAERRBAR in front of every arrive: the two
// edge warps of a CTA spent half their time there and the whole wavefront ran at their pace (profiles/r2_vwave_kernels.md).
__device__ __forceinline__ void vw_mbar_arrive_remote(uint32_t rbar) {
    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(rbar) : "memory");
}
__device__ __forceinline__ void vw_mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "VW_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra VW_DONE_%=;\n\t"
        "bra VW_WAIT_%=;\n\t"
        "VW_DONE_%=:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void vw_bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void vw_bulk_s2g(void* dst, uint32_t src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ uint32_t vw_mapa(uint32_t local_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void vw_st_async(uint32_t raddr, uint32_t v, uint32_t rbar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];"
                 ::"r"(raddr), "r"(v), "r"(rbar) : "memory");
}
// One-lane operations as PREDICATED instructions instead of `if (lane == 0)` branches: a divergent region makes the whole warp
// wait at its reconvergence point until lane 0's barrier instruction has gone through (measured: ~180 cycles per
// `if (lane == 0) mbarrier.arrive`, six such regions per row); a predicated instruction is just issued.
__device__ __forceinline__ void vw_mbar_arrive_if(uint32_t bar, bool p) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %1, 0;\n\t@q mbarrier.arrive.shared::cta.b64 _, [%0];\n\t}" ::"r"(bar), "r"((uint32_t)p) : "memory");
}
__device__ __forceinline__ void vw_mbar_arrive_remote_if(uint32_t rbar, bool p) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %1, 0;\n\t@q mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];\n\t}" ::"r"(rbar), "r"((uint32_t)p) : "memory");
}
__device__ __forceinline__ void vw_mbar_expect_tx_if(uint32_t bar, uint32_t bytes, bool p) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %2, 0;\n\t@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t}" ::"r"(bar), "r"(bytes), "r"((uint32_t)p) : "memory");
}
__device__ __forceinline__ void vw_st_async_if(uint32_t raddr, uint32_t v, uint32_t rbar, bool p) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %3, 0;\n\t@q st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];\n\t}"
                 ::"r"(raddr), "r"(v), "r"(rbar), "r"((uint32_t)p) : "memory");
}
__device__ __forceinline__ void vw_st_shared_if(uint32_t addr, uint32_t v, bool p) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %2, 0;\n\t@q st.shared.b32 [%0], %1;\n\t}" ::"r"(addr), "r"(v), "r"((uint32_t)p) : "memory");
}
template <int NP> __device__ __forceinline__ void vw_st_async_vec(uint32_t raddr, const uint32_t (&v)[NP], uint32_t rbar);
template <> __device__ __forceinline__ void vw_st_async_vec<1>(uint32_t raddr, const uint32_t (&v)[1], uint32_t rbar) {
    vw_st_async(raddr, v[0], rbar);
}
template <> __device__ __forceinline__ void vw_st_async_vec<2>(uint32_t raddr, const uint32_t (&v)[2], uint32_t rbar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.b32 [%0], {%1, %2}, [%3];"
                 ::"r"(raddr), "r"(v[0]), "r"(v[1]), "r"(rbar) : "memory");
}
template <> __device__ __forceinline__ void vw_st_async_vec<4>(uint32_t raddr, const uint32_t (&v)[4], uint32_t rbar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];"
                 ::"r"(raddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(rbar) : "memory");
}

// a lane's NP words into a slot of this CTA's shared memory (address in the shared window)
template <int NP> __device__ __forceinline__ void vw_st_local_vec(uint32_t addr, const uint32_t (&v)[NP]);
template <> __device__ __forceinline__ void vw_st_local_vec<1>(uint32_t addr, const uint32_t (&v)[1]) {
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v[0]) : "memory");
}
template <> __device__ __forceinline__ void vw_st_local_vec<2>(uint32_t addr, const uint32_t (&v)[2]) {
    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(v[0]), "r"(v[1]) : "memory");
}
template <> __device__ __forceinline__ void vw_st_local_vec<4>(uint32_t addr, const uint32_t (&v)[4]) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]) : "memory");
}

// stage index of a double-buffered resource: a compile-time value when the row loop is unrolled by two (every stage offset
// an immediate), a register otherwise (one copy of the row body: half the instruction footprint)
template <int V> struct VwStageCt { __device__ __forceinline__ constexpr int get() const { return V; } };
struct VwStageRt { int v; __device__ __forceinline__ int get() const { return v; } };

template <int NP> struct VwVec;
template <> struct VwVec<1> { typedef uint32_t T; };
template <> struct VwVec<2> { typedef uint2 T; };
template <> struct VwVec<4> { typedef uint4 T; };
template <int NP> __device__ __forceinline__ void vw_unpack(const typename VwVec<NP>::T& v, uint32_t (&o)[NP]);
template <> __device__ __forceinline__ void vw_unpack<1>(const uint32_t& v, uint32_t (&o)[1]) { o[0] = v; }
template <> __device__ __forceinline__ void vw_unpack<2>(const uint2& v, uint32_t (&o)[2]) { o[0] = v.x; o[1] = v.y; }
template <> __device__ __forceinline__ void vw_unpack<4>(const uint4& v, uint32_t (&o)[4]) { o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w; }
template <int NP> __device__ __forceinline__ typename VwVec<NP>::T vw_pack(const uint32_t (&o)[NP]);
template <> __device__ __forceinline__ uint32_t vw_pack<1>(const uint32_t (&o)[1]) { return o[0]; }
template <> __device__ __forceinline__ uint2 vw_pack<2>(const uint32_t (&o)[2]) { return make_uint2(o[0], o[1]); }
template <> __device__ __forceinline__ uint4 vw_pack<4>(const uint32_t (&o)[4]) { return make_uint4(o[0], o[1], o[2], o[3]); }

// OpenCV's uniqueness test (modes SGBM / HH), see wta_not_unique in sgbm.cu; out of line, uniquenessRatio > 0 only
template <int NP>
__device__ __noinline__ bool vw_not_unique(typename VwVec<NP>::T wv, unsigned key, int uniq, unsigned dkey) {
    uint32_t w[NP];
    vw_unpack<NP>(wv, w);
    const int minS = (int)(key >> 8), best = (int)(key & 255u);
    bool rej = false;
#pragma unroll
    for (int q = 0; q < NP; q++) {
        const int s0 = (int)(w[q] & 0xffffu), s1 = (int)(w[q] >> 16);
        const int d0 = (int)dkey + 2 * q;
        if (s0 * (100 - uniq) < minS * 100 && abs(best - d0) > 1) rej = true;
        if (s1 * (100 - uniq) < minS * 100 && abs(best - d0 - 1) > 1) rej = true;
    }
    return __any_sync(0xffffffffu, rej) && minS < 32767;
}

// NP = D / 64 words per lane (D in {64, 128}); CPW = columns per warp
// LAST = false: pass 1 (rows top-down, columns left-to-right), S = sum of the four path costs (S is not read), written back
// LAST = true:  pass 2 (the volume mirrored in x and y), S += the four path costs, winner-takes-all on the finished
//               rows, S not written back
// FULL:         width1 is a multiple of CPW (every strip has CPW columns): all column offsets are immediates
//
// One row of a warp (row-time), in this order so that the left-to-right chain of the horizontal path moves on after
// about a fifth of a row-time (fill and drain of the wavefront: ~0.2 x warps row-times instead of 1 x warps):
//   left edge in  {H after the left neighbour's last column of THIS row, its A state after the PREVIOUS row}
//   H chain       CPW dependent steps; each column's cost is parked in shared memory for the S sum
//   left edge out {H after my last column, my last column's A state as it still is: after the previous row}
//   B, column 0   -> right edge out (the left neighbour needs it for its NEXT row, late in its row-time)
//   A columns, B columns 1 .. CPW-2, right edge in (the right neighbour's B state after the previous row), B column CPW-1
//   V + S sum (+ winner-takes-all keys) per column, epilogue, TMA store / loads
// PAIRED (D = 128, an even CPW >= 4): the A, V and B paths of columns p and p + CPW/2 run as one sgm_step_pair, so "column j"
// above reads "slot j" and the diagonal hand-off stays a register rename (A of slot p reads slot p-1, B reads slot p+1).  The
// edge slots of the neighbours carry one column in sgm_step's layout as before; the first and the last slot assemble their
// mixed input (A: the left neighbour's column and my column CPW/2 - 1; B: my column CPW/2, kept from before slot 0 moved
// on, and the right neighbour's column) with PRMTs.  V runs beside A on the same interleaved costs; the S sum adds A + B +
// V of both columns in the paired layout and splits it before the horizontal path's costs are added.  Odd CPW, and
// D = 64 / 256, keep one column per slot (sgm_step).
// NW = warps per CTA: 16 (128 registers per thread) up to D = 128, 8 (255 registers) at D = 256, where a column's state is
// 15 registers.  At D = 256 the neighbour slots are single-buffered (SB) and the last pass adds the horizontal path's
// costs into the S row in place (HIP): see vwave_warp_bytes.
template <int NP, int CPW, bool LAST, bool FULL, int NW>
__global__ void __launch_bounds__(NW * 32, 1) sgbm_vwave_kernel(const VWaveArgs a) {
    constexpr int VW_WARPS = NW;
    constexpr bool SB = NP > 2, HIP = NP > 2, ROLLH = NP > 2;
    typedef typename VwVec<NP>::T vec;
    constexpr uint32_t INF = 0x7fff7fffu;
    constexpr uint32_t B = 128u * NP;                      // bytes per pixel vector (D = 64 NP disparities)
    constexpr uint32_t rowb = (uint32_t)CPW * B, slot = B + 16;
    // Shared memory of a warp: two STAGE BLOCKS a fixed distance DELTA apart, each [C row | S row | 5 mbarriers | Lin: H slot,
    // A slot | Rin slot], so that every address that depends on the stage of a row is (one register: block base) + (a
    // compile-time offset) -- with the stage as a register (one copy of the row body) the addresses cost one toggle per
    // row instead of a multiply-add each.  Single-buffered slots (SB) live in block 0 only; block 1 is then [C | S | bars].
    constexpr uint32_t O_C = 0, O_S = rowb, O_BAR = 2 * rowb, O_LIN = 2 * rowb + 64, O_RIN = O_LIN + 2 * slot;
    constexpr uint32_t DELTA = vwave_delta(rowb, slot);
    constexpr uint32_t WBS = SB ? ((DELTA + 2 * rowb + 64 + 127u) & ~127u) : 2 * DELTA;   // both blocks
    constexpr uint32_t WB = WBS + (LAST && !HIP ? rowb : 0);                         // + the horizontal path's row
    constexpr int DIR = LAST ? -1 : 1;
    constexpr bool UNROLL2 = !LAST && NP <= 2;
    // the previous-row paths (A, V, B) of columns p and p + HP share words (sgm_step_pair); the horizontal chain cannot
    constexpr bool PAIRED = NP == 2 && CPW % 2 == 0 && CPW >= 4;
    constexpr int HP = CPW / 2, NS = PAIRED ? HP : CPW, NWD = PAIRED ? 4 : NP;
    extern __shared__ __align__(128) unsigned char vw_smem[];
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int CL = a.cluster;
    const int job = blockIdx.y;
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    const int lane = threadIdx.x & 31;
    const bool lane0 = lane == 0;
    const int width1 = a.width1, H = a.H;
    const int g = rank * VW_WARPS + warp;                  // strip number, left to right in pass coordinates
    const int u0 = g * CPW;                                // first column (pass coordinates) of this warp
    const int ncols = FULL ? (u0 < width1 ? CPW : 0) : max(0, min(CPW, width1 - u0));  // valid columns
    const int nstrips = (width1 + CPW - 1) / CPW;
    const bool has_left = g > 0, has_right = g + 1 < nstrips;
    // memory block of a row: image columns [xb, xb + ncols); pass column j <-> block column (DIR > 0 ? j : ncols - 1 - j)
    const int xb = DIR > 0 ? u0 : max(width1 - u0 - CPW, 0);
    unsigned char* wbase = vw_smem + (size_t)warp * WB;
    unsigned char* Hrow = wbase + WBS;                     // LAST && !HIP only: [rowb] the horizontal path's costs of the current row
    // barriers of a block, at O_BAR: +0 row landed (TMA) | +8 left slot (Lin) full | +16 right slot (Rin) full | +24 my
    // outgoing left-edge slot (in the right neighbour) free | +32 my outgoing right-edge slot (in the left neighbour) free
    constexpr uint32_t B_TMA = O_BAR, B_LF = O_BAR + 8, B_RF = O_BAR + 16, B_LE = O_BAR + 24, B_RE = O_BAR + 32;
    const char* Cg = (const char*)a.C[job];
    char* Sg = (char*)a.S[job];
    const int uniq = a.uniq[job];
    uint2* recg = a.rec[job];
    const unsigned dkey = (unsigned)(lane * 2 * NP);
    const unsigned dpair = dkey | ((dkey + 1u) << 8);

    if (lane == 0) {
        // a slot is filled either by plain stores + one arrive (same CTA) or by st.async bytes + the consumer's own
        // expect_tx arrive (neighbour CTA): one arrival per phase in both cases
        const uint32_t w0 = (uint32_t)__cvta_generic_to_shared(wbase);
        for (int i = 0; i < 5; i++) { vw_mbar_init(w0 + O_BAR + 8 * i, 1); vw_mbar_init(w0 + DELTA + O_BAR + 8 * i, 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    cluster.sync();  // every warp's barriers exist before a neighbour signals them

    // where the edges go
    const bool left_remote = warp == 0 && rank > 0;                   // my left neighbour lives in the previous CTA
    const bool right_remote = warp == VW_WARPS - 1 && rank < CL - 1;  // my right neighbour lives in the next CTA
    // outgoing left-edge data (H, A) -> right neighbour's Lin; outgoing right-edge data (B) -> left neighbour's Rin.
    // All as shared-window addresses: the same 32-bit arithmetic serves local (shared::cta) and remote (shared::cluster).
    uint32_t nbR = 0, nbL = 0;   // block 0 of the right / left neighbour's shared memory (this CTA's or, mapped, the next one's)
    const uint32_t wbase_s = (uint32_t)__cvta_generic_to_shared(wbase);
    if (has_right) {
        const uint32_t nb = right_remote ? vw_mapa((uint32_t)__cvta_generic_to_shared(vw_smem), (uint32_t)(rank + 1)) : wbase_s + WB;
        nbR = nb;   // its Lin (+ O_LIN) and Lin-full barrier (+ B_LF) take my {H, A}; its B_RE is where I signal "Rin slot read"
    }
    if (has_left) {
        const uint32_t nb = left_remote ? vw_mapa((uint32_t)__cvta_generic_to_shared(vw_smem) + (VW_WARPS - 1) * WB, (uint32_t)(rank - 1))
                                        : wbase_s - WB;
        nbL = nb;   // its Rin (+ O_RIN) and Rin-full barrier (+ B_RF) take my B; its B_LE is where I signal "Lin slot read"
    }

    auto load_row = [&](int it) {  // lane 0: C (and S) of my columns of the it-th processed row into stage it & 1
        const int row = DIR > 0 ? it : H - 1 - it;
        const uint32_t bytes = (uint32_t)ncols * B;
        const uint32_t blk = wbase_s + (uint32_t)(it & 1) * DELTA, bar = blk + B_TMA;
        const size_t off = ((size_t)row * width1 + xb) * B;
        vw_mbar_expect_tx(bar, LAST ? 2 * bytes : bytes);
        vw_bulk_g2s(blk + O_C, Cg + off, bytes, bar);
        if (LAST) vw_bulk_g2s(blk + O_S, Sg + off, bytes, bar);
    };
    const bool active = ncols > 0;
    if (active && lane == 0) {
        load_row(0);
        if (H > 1) load_row(1);
    }

    // path state: A = diagonal fed from the left neighbour column, V = vertical, Bp = diagonal fed from the right.
    // PAIRED: slot p holds columns p (low halves) and p + HP (high halves) in sgm_step_pair's layout, 4 words per lane;
    // otherwise slot j is column j, NP words in sgm_step's layout.
    uint32_t LA[NS][NWD], LV[NS][NWD], LB[NS][NWD];
    uint32_t mA[NS], mV[NS], mB[NS];
#pragma unroll
    for (int j = 0; j < NS; j++) {
#pragma unroll
        for (int k = 0; k < NWD; k++) { LA[j][k] = 0; LV[j][k] = 0; LB[j][k] = 0; }
        mA[j] = 0; mV[j] = 0; mB[j] = 0;
    }
    const uint32_t p1x2 = (uint32_t)a.P1 * 0x10001u;
    const uint32_t k2 = (0x10000u - (uint32_t)a.P2) * 0x10001u;
    const SgmLane sl = sgm_lane_init(lane, a.zero);
    // block column (in vectors of the warp: x 32 lanes) of pass column j
    int jbr[FULL ? 1 : CPW];
    if (!FULL) {
#pragma unroll
        for (int j = 0; j < CPW; j++) jbr[FULL ? 0 : j] = j < ncols ? (DIR > 0 ? j : ncols - 1 - j) : 0;
    }
    auto JB = [&](int j) -> int { return FULL ? (DIR > 0 ? j : CPW - 1 - j) : jbr[FULL ? 0 : j]; };
    auto valid = [&](int j) -> bool { return FULL || j < ncols; };

    // one row; ST = it & 1.  Pass 1 unrolls the row loop by two (ST a compile-time value).  The last pass keeps ONE copy of
    // its longer body: two copies (42 KB of code, 16 warps per SM all at different places of it) ran with 13 % of the
    // stall samples on instruction fetch (profiles/r2_vwave_kernels.md).
    auto do_row = [&](const int it, auto st_tag) {
        const int ST = st_tag.get();
        const uint32_t ph = (uint32_t)((it >> 1) & 1);      // phase of the it-th use of a double-buffered resource
        // neighbour slots: stage and phase of this row's use, and what a producer waits for before it reuses a stage (the
        // consumer's "free" signal for the previous content: two rows back when double-buffered, else the previous row)
        const int SS = SB ? 0 : ST;
        const uint32_t sph = SB ? (uint32_t)(it & 1) : ph;
        const bool reuse = SB ? it >= 1 : it >= 2;
        const uint32_t fph = sph ^ 1u;
        // block bases: this row's stage (C, S, TMA barrier), the slots' stage (SS), the stage of the right neighbour's previous
        // row (SE, right edge in); the same offsets in the neighbours' shared memory
        const uint32_t so = (uint32_t)ST * DELTA, sso = (uint32_t)SS * DELTA;
        unsigned char* blk = wbase + so;
        const uint32_t blk_s = wbase_s + so, sblk_s = wbase_s + sso;
        vw_mbar_wait(blk_s + B_TMA, ph);
        const vec* cs = (const vec*)(blk + O_C) + lane;   // cs[JB(j) * 32]: pass column j
        vec* ss = (vec*)(blk + O_S) + lane;
        vec* hs = (vec*)(LAST && !HIP ? Hrow : blk + O_S) + lane;  // where the horizontal path parks its costs
        uint32_t Cw[NP];
        // ---- left edge in
        uint32_t LH[NP], mH = 0, inA[NP], inAm = 0;
#pragma unroll
        for (int k = 0; k < NP; k++) { LH[k] = 0; inA[k] = 0; }
        if (has_left) {
            const uint32_t hb = sblk_s + B_LF;
            if (left_remote) {
                vw_mbar_expect_tx_if(hb, 2 * (B + 4u), lane0);
                __syncwarp();
            }
            vw_mbar_wait(hb, sph);
            const unsigned char* q = wbase + sso + O_LIN;
            vw_unpack<NP>(*(const vec*)(q + lane * sizeof(vec)), LH);
            mH = *(const uint32_t*)(q + B);
            vw_unpack<NP>(*(const vec*)(q + slot + lane * sizeof(vec)), inA);
            inAm = *(const uint32_t*)(q + slot + B);
            __syncwarp();
            // the "slot free" arrive carries a (zero) term computed from what was just read: it cannot issue before the
            // loads have returned, which is all the relaxed remote form needs
            const uint32_t dep = (LH[0] | inA[0] | mH | inAm) & sl.zero;
            if (left_remote) vw_mbar_arrive_remote_if(nbL + sso + B_LE + dep, lane0); else vw_mbar_arrive_if(nbL + sso + B_LE, lane0);
        }
        // ---- horizontal path: along the row through my columns
        auto h_column = [&](const int jb, const bool ok) {   // jb: block column of the pass column; ok: it is inside the volume
            vw_unpack<NP>(cs[jb * 32], Cw);
            mH = sgm_step<NP>(LH, LH, mH, Cw, p1x2, k2, sl);
            if (LAST && HIP) {   // S row (landed with this row's C) += horizontal path, in place
                uint32_t Sw[NP];
                vw_unpack<NP>(hs[jb * 32], Sw);
#pragma unroll
                for (int k = 0; k < NP; k++) Sw[k] = __viaddmin_u16x2(Sw[k], LH[k], INF);
                if (ok) hs[jb * 32] = vw_pack<NP>(Sw);
            } else if (ok) hs[jb * 32] = vw_pack<NP>(LH);
        };
        if (ROLLH) {
            // the chain touches no per-column registers, so it can be a real loop: D = 256 needs the instruction footprint
            // (the unrolled last pass was 48 KB of code and ran with 52 % of its stall samples on instruction fetch)
#pragma unroll 2
            for (int j = 0; j < CPW; j++) {
                const bool ok = FULL || j < ncols;
                const int jb = FULL ? (DIR > 0 ? j : CPW - 1 - j) : (ok ? (DIR > 0 ? j : ncols - 1 - j) : 0);
                h_column(jb, ok);
            }
        } else {
#pragma unroll
            for (int j = 0; j < CPW; j++) h_column(JB(j), valid(j));
        }
        // PAIRED: one column of a slot in sgm_step's layout (k = 0: the low halves, 1: the high halves).  The minimum words
        // that go with an edge slot stay packed (min of column p | min of column p + HP << 16): the consumer picks its half.
        auto half_of = [&](const uint32_t (&w)[NWD], int k, uint32_t (&o)[NP]) {
            const uint32_t sel = k ? 0x7632u : 0x5410u;
            o[0] = __byte_perm(w[0], w[1 % NWD], sel);
            o[NP - 1] = __byte_perm(w[2 % NWD], w[3 % NWD], sel);
        };
        // PAIRED: the costs of every slot, interleaved once per row (below) and shared by its A, V and B steps
        [[maybe_unused]] uint32_t Cs[PAIRED ? NS : 1][NWD];
        auto c_slot = [&](int p, uint32_t (&Cp)[NWD]) {
            if constexpr (PAIRED) {
#pragma unroll
                for (int k = 0; k < NWD; k++) Cp[k] = Cs[p][k];
            } else {
                vw_unpack<NP>(cs[JB(p) * 32], Cp);
            }
        };
        auto step = [&](uint32_t (&O)[NWD], const uint32_t (&I)[NWD], uint32_t minI2, const uint32_t (&Cp)[NWD]) -> uint32_t {
            if constexpr (PAIRED) return sgm_step_pair(O, I, minI2, Cp, p1x2, k2, sl);
            else return sgm_step<NP>(O, I, minI2, Cp, p1x2, k2, sl);
        };
        // ---- left edge out: my last column's A state as it still is (after the previous row)
        if (has_right) {
            uint32_t eA[NP], emA;
            if constexpr (PAIRED) { half_of(LA[HP - 1], 1, eA); emA = mA[HP - 1]; }   // column CPW - 1: the high half
            else {
#pragma unroll
                for (int k = 0; k < NP; k++) eA[k] = LA[CPW - 1][k % NWD];
                emA = mA[CPW - 1];
            }
            if (reuse) vw_mbar_wait(sblk_s + B_LE, fph);
            const uint32_t q = nbR + sso + O_LIN, rb = nbR + sso + B_LF;
            if (!right_remote) {
                vw_st_local_vec<NP>(q + lane * (uint32_t)sizeof(vec), LH);
                vw_st_local_vec<NP>(q + slot + lane * (uint32_t)sizeof(vec), eA);
                vw_st_shared_if(q + B, mH, lane0);
                vw_st_shared_if(q + slot + B, emA, lane0);
                __syncwarp();
                vw_mbar_arrive_if(rb, lane0);
            } else {
                vw_st_async_vec<NP>(q + lane * (uint32_t)sizeof(vec), LH, rb);
                vw_st_async_vec<NP>(q + slot + lane * (uint32_t)sizeof(vec), eA, rb);
                vw_st_async_if(q + B, mH, rb, lane0);
                vw_st_async_if(q + slot + B, emA, rb, lane0);
            }
        }
        // A of slot 0 reads (the left neighbour's last column, my column HP - 1): assembled before slot HP - 1 moves on
        uint32_t inA0[NWD], inA0m;
        if constexpr (PAIRED) {
            inA0[0] = __byte_perm(inA[0], LA[HP - 1][0], 0x5410); inA0[1] = __byte_perm(inA[0], LA[HP - 1][1], 0x5432);
            inA0[2] = __byte_perm(inA[1], LA[HP - 1][2], 0x5410); inA0[3] = __byte_perm(inA[1], LA[HP - 1][3], 0x5432);
            inA0m = __byte_perm(inAm, mA[HP - 1], 0x5432);
        } else {
#pragma unroll
            for (int k = 0; k < NWD; k++) inA0[k] = inA[k % NP];
            inA0m = inAm;
        }
        // ---- B path, first column (slot 0), and right edge out.  PAIRED: B of the last slot reads (column HP, the right
        // neighbour's first column); column HP is the high half of slot 0, kept here as it was after the previous row.
        [[maybe_unused]] uint32_t svB[NP], svBm = 0;
        if constexpr (PAIRED) { half_of(LB[0], 1, svB); svBm = mB[0]; }
        if constexpr (PAIRED) {
#pragma unroll
            for (int p = 0; p < NS; p++) {
                uint32_t ca[NP], cb[NP];
                vw_unpack<NP>(cs[JB(p) * 32], ca);
                vw_unpack<NP>(cs[JB(p + HP) * 32], cb);
                Cs[p][0] = __byte_perm(ca[0], cb[0], 0x5410); Cs[p][1] = __byte_perm(ca[0], cb[0], 0x7632);
                Cs[p][2] = __byte_perm(ca[1], cb[1], 0x5410); Cs[p][3] = __byte_perm(ca[1], cb[1], 0x7632);
            }
        }
        uint32_t Cp[NWD];
        c_slot(0, Cp);
        mB[0] = step(LB[0], LB[1], mB[1], Cp);
        if (has_left && it + 1 < H) {
            uint32_t eB[NP], emB;
            if constexpr (PAIRED) { half_of(LB[0], 0, eB); emB = mB[0]; }   // column 0: the low half
            else {
#pragma unroll
                for (int k = 0; k < NP; k++) eB[k] = LB[0][k % NWD];
                emB = mB[0];
            }
            if (reuse) vw_mbar_wait(sblk_s + B_RE, fph);                // the neighbour has read the slot's previous content
            const uint32_t q = nbL + sso + O_RIN, rb = nbL + sso + B_RF;
            if (!left_remote) {
                vw_st_local_vec<NP>(q + lane * (uint32_t)sizeof(vec), eB);
                vw_st_shared_if(q + B, emB, lane0);
                __syncwarp();
                vw_mbar_arrive_if(rb, lane0);
            } else {
                vw_st_async_vec<NP>(q + lane * (uint32_t)sizeof(vec), eB, rb);
                vw_st_async_if(q + B, emB, rb, lane0);
            }
        }
        // ---- diagonal A (fed from the left): in place, right to left (slot j reads slot j-1's old state)
#pragma unroll
        for (int j = NS - 1; j >= 1; j--) {
            c_slot(j, Cp);
            mA[j] = step(LA[j], LA[j - 1], mA[j - 1], Cp);
            if (PAIRED) mV[j] = step(LV[j], LV[j], mV[j], Cp);   // (PAIRED: V shares the interleaved costs with A)
        }
        c_slot(0, Cp);
        mA[0] = step(LA[0], inA0, inA0m, Cp);
        if (PAIRED) mV[0] = step(LV[0], LV[0], mV[0], Cp);
        // ---- diagonal B (fed from the right): in place, left to right; the last slot needs the right neighbour's state
#pragma unroll
        for (int j = 1; j < NS - 1; j++) {
            c_slot(j, Cp);
            mB[j] = step(LB[j], LB[j + 1], mB[j + 1], Cp);
        }
        {
            uint32_t inB[NP], inBm = 0;
#pragma unroll
            for (int k = 0; k < NP; k++) inB[k] = 0;
            if (has_right && it > 0) {  // B state of the neighbour's first column after row it - 1 (its stage and phase)
                const uint32_t seo = SB ? 0u : DELTA - so;   // the other stage's block
                const uint32_t hb = wbase_s + seo + B_RF;
                if (right_remote) {
                    vw_mbar_expect_tx_if(hb, B + 4u, lane0);
                    __syncwarp();
                }
                vw_mbar_wait(hb, SB ? (uint32_t)((it - 1) & 1) : (uint32_t)(((it - 1) >> 1) & 1));
                const unsigned char* q = wbase + seo + O_RIN;
                vw_unpack<NP>(*(const vec*)(q + lane * sizeof(vec)), inB);
                inBm = *(const uint32_t*)(q + B);
                __syncwarp();
                const uint32_t dep = (inB[0] | inBm) & sl.zero;
                if (right_remote) vw_mbar_arrive_remote_if(nbR + seo + B_RE + dep, lane0); else vw_mbar_arrive_if(nbR + seo + B_RE, lane0);
            }
            uint32_t inBL[NWD], inBLm;
            if constexpr (PAIRED) {
                inBL[0] = __byte_perm(svB[0], inB[0], 0x5410); inBL[1] = __byte_perm(svB[0], inB[0], 0x7632);
                inBL[2] = __byte_perm(svB[1], inB[1], 0x5410); inBL[3] = __byte_perm(svB[1], inB[1], 0x7632);
                inBLm = __byte_perm(svBm, inBm, 0x5432);
            } else {
#pragma unroll
                for (int k = 0; k < NWD; k++) inBL[k] = inB[k % NP];
                inBLm = inBm;
            }
            c_slot(NS - 1, Cp);
            mB[NS - 1] = step(LB[NS - 1], inBL, inBLm, Cp);
        }
        if (!FULL && ncols < CPW) {
            // columns outside the volume: their state must read as "no predecessor" (0) for the last valid column
#pragma unroll
            for (int j = 0; j < NS; j++) {
                if constexpr (PAIRED) {   // slot j holds columns j and j + HP
                    const uint32_t keep = (j < ncols ? 0xffffu : 0u) | (j + HP < ncols ? 0xffff0000u : 0u);
#pragma unroll
                    for (int k = 0; k < NWD; k++) LB[j][k] &= keep;
                    mB[j] &= keep;
                } else if (j >= ncols) {
#pragma unroll
                    for (int k = 0; k < NWD; k++) LB[j][k] = 0;
                    mB[j] = 0;
                }
            }
        }
        // ---- vertical path + S row
        unsigned wkey = 0xffffffffu;
        bool wrej = false;
        auto wta_column = [&](const uint32_t (&Sw)[NP], const int j) {   // arg-min key (+ uniqueness) of pass column j -> lane j
            unsigned key = 0xffffffffu;
#pragma unroll
            for (int k = 0; k < NP; k++) {
                const unsigned dk = dpair + 0x0202u * (unsigned)k;
                key = min(key, min(__byte_perm(Sw[k], dk, 0x7104), __byte_perm(Sw[k], dk, 0x7325)));
            }
            key = __reduce_min_sync(0xffffffffu, key);
            bool rej = false;
            if (uniq > 0) rej = vw_not_unique<NP>(vw_pack<NP>(Sw), key, uniq, dkey);
            if (lane == j) { wkey = key; wrej = rej; }
        };
#pragma unroll
        for (int j = 0; j < NS; j++) {
            if constexpr (PAIRED) {
                // A + B + V of both columns at once, then per column + H (+ S): all terms are non-negative and at most
                // 32767, so the saturating adds give min(sum, 32767) in any order
                uint32_t s3[NWD];
#pragma unroll
                for (int k = 0; k < NWD; k++) s3[k] = __viaddmin_u16x2(__viaddmin_u16x2(LA[j][k], LB[j][k], INF), LV[j][k], INF);
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    const int jc = j + h * HP;
                    uint32_t Sw[NP], Hw[NP];
                    half_of(s3, h, Sw);
                    vw_unpack<NP>(hs[JB(jc) * 32], Hw);
#pragma unroll
                    for (int k = 0; k < NP; k++) Sw[k] = __viaddmin_u16x2(Sw[k], Hw[k], INF);
                    if (LAST) {
                        uint32_t Sr[NP];
                        vw_unpack<NP>(ss[JB(jc) * 32], Sr);
#pragma unroll
                        for (int k = 0; k < NP; k++) Sw[k] = __viaddmin_u16x2(Sr[k], Sw[k], INF);
                    }
                    if (valid(jc)) ss[JB(jc) * 32] = vw_pack<NP>(Sw);
                    if (LAST) wta_column(Sw, jc);
                }
            } else {
                c_slot(j, Cp);
                mV[j] = step(LV[j], LV[j], mV[j], Cp);
                uint32_t Sw[NP], Hw[NP];
                if (!(LAST && HIP)) vw_unpack<NP>(hs[JB(j) * 32], Hw);
                if (LAST) vw_unpack<NP>(ss[JB(j) * 32], Sw);
#pragma unroll
                for (int k = 0; k < NP; k++) {
                    uint32_t s3 = __viaddmin_u16x2(LA[j][k % NWD], LB[j][k % NWD], INF);
                    if (LAST && HIP) {
                        s3 = __viaddmin_u16x2(s3, LV[j][k % NWD], INF);
                    } else {
                        const uint32_t s4 = __viaddmin_u16x2(LV[j][k % NWD], Hw[k], INF);
                        s3 = __viaddmin_u16x2(s3, s4, INF);
                    }
                    Sw[k] = LAST ? __viaddmin_u16x2(Sw[k], s3, INF) : s3;
                }
                if (valid(j)) ss[JB(j) * 32] = vw_pack<NP>(Sw);  // columns outside the volume alias block column 0: never stored
                if (LAST && !ROLLH) wta_column(Sw, j);
            }
        }
        if (LAST && ROLLH) {
            // winner-takes-all keys from the finished S row in shared memory, as a real loop (instruction footprint, see
            // the horizontal chain); every lane reads back what it stored itself
#pragma unroll 4
            for (int j = 0; j < (FULL ? CPW : ncols); j++) {   // (four columns in flight: the reductions overlap)
                uint32_t Sw[NP];
                vw_unpack<NP>(ss[(DIR > 0 ? j : (FULL ? CPW : ncols) - 1 - j) * 32], Sw);
                wta_column(Sw, j);
            }
        }
        if (LAST) {
            // One record per finished pixel: the winner key and the two S neighbours of the minimum.  The disp2 vote, the
            // sub-pixel division and the store of the raw disparity are vw_finish_kernel's job (one thread per pixel): here
            // 9 of 32 lanes ran ~100 dependent instructions per row, 19 % of the pass's stall samples.
            __syncwarp();
            if (lane < ncols) {
                const int u = u0 + lane;                               // pass column of lane's pixel
                const int y = DIR > 0 ? it : H - 1 - it;
                const int x = DIR > 0 ? u : width1 - 1 - u;
                const int d = (int)(wkey & 255u);
                uint2 rec = make_uint2(0xffffffffu, 0u);
                if ((wkey >> 8) < 32767u && !wrej) {
                    const int jbl = DIR > 0 ? lane : ncols - 1 - lane;
                    const uint16_t* Sp = (const uint16_t*)(blk + O_S + (size_t)jbl * B);
                    rec = make_uint2(wkey, (unsigned)Sp[max(d - 1, 0)] | ((unsigned)Sp[min(d + 1, 64 * NP - 1)] << 16));
                }
                recg[(size_t)y * width1 + x] = rec;
            }
        }
        // ---- S row out (first pass), next-but-one row in
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
            if (!LAST) {
                const int row = DIR > 0 ? it : H - 1 - it;
                vw_bulk_s2g(Sg + ((size_t)row * width1 + xb) * B, blk_s + O_S, (uint32_t)ncols * B);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                // the other stage's store (row it - 1) must have read its buffer before row it + 1 writes into it
                asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            }
            if (it + 2 < H) load_row(it + 2);
        }
        __syncwarp();
    };
    if (active) {
        if (UNROLL2) {
            int it = 0;
            for (; it + 1 < H; it += 2) {
                do_row(it, VwStageCt<0>());
                do_row(it + 1, VwStageCt<1>());
            }
            if (it < H) do_row(it, VwStageCt<0>());
        } else {
#pragma unroll 1
            for (int it = 0; it < H; it++) do_row(it, VwStageRt{it & 1});
        }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    cluster.sync();  // no CTA exits while a neighbour may still write into its shared memory or signal its barriers
}

// one launch of a given instantiation (all volumes of `a`: grid (cluster, jobs))
template <int NP, int CPW, int NW>
static int vwave_launch_shape(Lane& L, const VWaveArgs& a, int nj, bool last, bool full, size_t smem) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(a.cluster, nj);
    cfg.blockDim = dim3(NW * 32);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = L.stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = a.cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
#define VW_LAUNCH(KERN)                                                                                               \
    {                                                                                                                 \
        L3D_CHECK(L, cudaFuncSetAttribute(KERN, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));             \
        L3D_CHECK(L, cudaFuncSetAttribute(KERN, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));                  \
        if (!dbg_skip("sgbm_vwave_kernel")) L3D_CHECK(L, cudaLaunchKernelEx(&cfg, KERN, a));                          \
        L.launches++;                                                                                                 \
    }
    if (last && full) VW_LAUNCH((sgbm_vwave_kernel<NP, CPW, true, true, NW>))
    else if (last) VW_LAUNCH((sgbm_vwave_kernel<NP, CPW, true, false, NW>))
    else if (full) VW_LAUNCH((sgbm_vwave_kernel<NP, CPW, false, true, NW>))
    else VW_LAUNCH((sgbm_vwave_kernel<NP, CPW, false, false, NW>))
#undef VW_LAUNCH
    return L3D_OK;
}

// D = 256 instantiations live in a translation unit of their own (sgbm_vwave256.cu: 255-register kernels, slow to compile)
int vwave_launch_256(Lane& L, const VWaveArgs& a, int cpw, int nj, bool last, bool full, size_t smem);

}  // namespace l3d
