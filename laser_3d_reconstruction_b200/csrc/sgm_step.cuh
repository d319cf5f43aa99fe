// sgm_step.cuh -- one semi-global-matching path step for the disparities a lane holds (shared by the aggregation
// kernels of sgbm.cu, sgbm_hrow.cu and sgbm_vgroup.cu; cv2.StereoSGBM modes SGBM / HH / HH4 / 3WAY, SURVEY A4).
//
// A warp owns one pixel's disparity range, lane l holds 2*NP consecutive disparities as NP packed u16x2 words.
// sgm_step_pair (below) runs two independent D = 128 recurrences in the two halves of the words instead: no funnel words,
// no half-combine, 15 ALU-pipe instructions per step of the pair where two sgm_step<2> take 24.
// With delta = min_d(I) + P2 the step is
//     T[d] = min(I[d], I[d-1] + P1, I[d+1] + P1)          (I + P1 once per word on the FMA pipe, one VIMNMX3.U16x2)
//     O[d] = min(T[d] + (C[d] - delta), C[d])             (one VIADD.16x2, one VIADDMNMX.U16x2)
// which is OpenCV's  C + min(L[d], L[d+-1] + P1, delta) - delta.  Only the last two operations wait for the
// warp-wide minimum of the previous step, so the loop-carried chain through the reduction is
// CREDUX -> IMAD -> VIADDMNMX -> VIADD -> (min tree) -> CREDUX; the neighbour exchange (SHFL, PRMT, two VIADDMNMX) runs
// beside it.  -delta and C - delta are taken modulo 2^16; T + C - delta lies in [0, 2^16) because T >= min(I), delta =
// min(I) + P2 and C >= P2 (OpenCV's C carries P2), so the wrapped sum is the exact value and the unsigned minimum with C
// is the step's result; no zero operand is needed (the earlier form C + min(T - delta, 0) needed one: see below).
// I + P1 < 2^16 unsigned.
//
// Pipe balance (sm_100: the integer ALU pipe and the FMA pipe each accept one warp instruction every second cycle
// per SM sub-partition, so an all-ALU instruction stream tops out at half the issue rate; the cluster-fused
// aggregation kernel sits at ~80 % of the ALU pipe).  What this header does about it:
//   * a literal 0 as the third operand of VIADDMNMX makes ptxas build the zero with a PRMT in front of EVERY use (one
//     more ALU op per word: 2 of 17 per step at D = 128); the zero therefore comes in as a register whose value the
//     compiler cannot see (a kernel parameter);
//   * -(min + P2) is a multiply-add with an opaque -1 (FMA pipe) instead of an IADD3;
//   * the d-1 / d+1 neighbour words are funnel shifts of adjacent words; dm1 of word k+1 and dp1 of word k are the
//     same word, so a step needs NP + 1 of them.  The two that contain a neighbour lane's halves stay PRMTs (lanes 0
//     and 31 use a selector that feeds the word's own value into the missing slot -- L[d] + P1 - delta >= L[d] - delta
//     never wins); with FMAFUNNEL the NP - 1 interior ones become (x << 16) + (y >> 16) = IMAD(x, 65536,
//     IMAD.HI(y, 65536)) with the multiplier in a register, which ptxas keeps on the FMA pipe (tools/ubench/sgmstep.cu
//     measures all forms);
//   * I + P1 is carry-free in both halves (I + P1 < 2^16), so it is ONE 32-bit multiply-add per word with an opaque
//     multiplier 1 (FMA pipe); the neighbour words are funnelled from the sums and T is a single three-input minimum
//     instead of two add-min instructions: 12 instead of 14 ALU-pipe instructions per step at D = 128 (ubench: 30.0 ->
//     28.7 cycles per step and sub-partition; 50.9 -> 45.7 at D = 256).  Moving C + min(T - delta, 0) to the FMA pipe as
//     min(T, delta) + (C - delta) was measured too (30.4): two more IMADs per word cost more than the ALU slot they free.
#pragma once
#include <cstdint>

namespace l3d {

// loop-invariant per-lane operands of sgm_step
struct SgmLane {
    uint32_t selA, selB;  // byte-permute selectors of the edge funnel words (lane 0 / lane 31 specials)
    uint32_t zero;        // 0, opaque
    uint32_t neg1;        // 0xffffffff, opaque
    uint32_t m64k;        // 65536, opaque
    uint32_t one;         // 1, opaque
    uint32_t upm, upa;    // sgm_step_pair: the d-1 word from the lane below is x * upm + upa (lane 0: all ones, never wins)
    uint32_t dnm, dna;    // sgm_step_pair: the d+1 word from the lane above is x * dnm + dna (lane 31: all ones)
};
// zero_param = 0: a value the compiler cannot see (kernel parameter)
__device__ __forceinline__ SgmLane sgm_lane_init(int lane, uint32_t zero_param) {
    SgmLane s;
    s.selA = lane == 0 ? 0x5454u : 0x5432u;
    s.selB = lane == 31 ? 0x3232u : 0x5432u;
    s.zero = zero_param; s.neg1 = ~zero_param; s.m64k = zero_param + 65536u; s.one = zero_param + 1u;
    s.upm = zero_param + (lane == 0 ? 0u : 1u); s.upa = lane == 0 ? ~zero_param : zero_param;
    s.dnm = zero_param + (lane == 31 ? 0u : 1u); s.dna = lane == 31 ? ~zero_param : zero_param;
    return s;
}

__device__ __forceinline__ uint32_t sgm_madlo(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t sgm_mulhi(uint32_t a, uint32_t b) {
    uint32_t d;
    asm("mul.hi.u32 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
    return d;
}

// k2 = (0x10000 - P2) * 0x10001, p1x2 = P1 * 0x10001; k2 - minI2 cannot carry between the halves (minI <= 32767,
// P1 < P2 <= 16000).  In and out may be the same registers (every output word is computed
// before any is stored).  Returns the warp-wide minimum of O in both halves.
// FULL = false: lanes with `active` == false hold no disparities (D < 64 * NP); they keep O = MAX_COST so that neither
// the neighbour exchange nor the min-reduction sees them.
template <int NP, bool FMAFUNNEL = false, bool FULL = true>
__device__ __forceinline__ uint32_t sgm_step(uint32_t (&O)[NP], const uint32_t (&I)[NP], uint32_t minI2,
                                             const uint32_t (&Cv)[NP], uint32_t p1x2, uint32_t k2, const SgmLane& s,
                                             bool active = true) {
    static_assert(NP == 1 || NP == 2 || NP == 4 || NP == 8, "sgm_step: the warp minimum covers NP = 1, 2, 4 and 8 words");
    uint32_t Ip[NP];                                    // I + P1, both halves (no carry: I + P1 < 2^16)
#pragma unroll
    for (int k = 0; k < NP; k++) Ip[k] = sgm_madlo(I[k], s.one, p1x2);
    const uint32_t up = __shfl_up_sync(0xffffffffu, Ip[NP - 1], 1);
    const uint32_t dn = __shfl_down_sync(0xffffffffu, Ip[0], 1);
    const uint32_t nd2 = sgm_madlo(minI2, s.neg1, k2);   // -(minI + P2) mod 2^16, both halves
    uint32_t F[NP + 1];                                  // F[k] = (Ip[k-1] >> 16) | (Ip[k] << 16): dm1 of word k, dp1 of word k-1
    F[0] = __byte_perm(up, Ip[0], s.selA);
    F[NP] = __byte_perm(Ip[NP - 1], dn, s.selB);
#pragma unroll
    for (int k = 1; k < NP; k++)
        F[k] = FMAFUNNEL ? sgm_madlo(Ip[k], s.m64k, sgm_mulhi(Ip[k - 1], s.m64k)) : __byte_perm(Ip[k - 1], Ip[k], 0x5432);
    uint32_t Ln[NP];
#pragma unroll
    for (int k = 0; k < NP; k++) {
        const uint32_t t = __vimin3_u16x2(I[k], F[k], F[k + 1]);
        Ln[k] = __viaddmin_u16x2(t, __vadd2(Cv[k], nd2), Cv[k]);  // min(T + (C - delta), C), all modulo 2^16 (see above)
        if (!FULL && !active) Ln[k] = 0x7fff7fffu;
    }
    uint32_t mn = Ln[0];
    if (NP == 2) mn = __vminu2(Ln[0], Ln[1]);
    if (NP == 4) mn = __vimin3_u16x2(__vminu2(Ln[0], Ln[1]), Ln[2], Ln[3]);
    if constexpr (NP == 8)
        mn = __vimin3_u16x2(__vimin3_u16x2(Ln[0], Ln[1], Ln[2]), __vimin3_u16x2(Ln[3], Ln[4], Ln[5]), __vminu2(Ln[6], Ln[7]));
#pragma unroll
    for (int k = 0; k < NP; k++) O[k] = Ln[k];
    mn = __vminu2(mn, __byte_perm(mn, mn, 0x1032));  // both halves = min of the two
    return __reduce_min_sync(0xffffffffu, mn);        // packed halves are equal, so the u32 min is the packed min
}

// Two independent D = 128 recurrences at once (the paired form): word k of lane l holds disparity 4l + k of recurrence
// a in its low half and of recurrence b in its high half, so the d-1 / d+1 neighbours of word k are words k-1 / k+1 and
// only words 0 and 3 take one from the next lane (SHFL up / down; lanes 0 and 31 put all ones there through a
// multiply-add with per-lane constants, FMA pipe).  The per-half arithmetic is sgm_step's.  minI2 and the result are
// (min a | min b << 16): the four-word min tree gives the two per-lane minima directly, the warp takes them with two
// CREDUX.MIN -- one on m (high half: min of the high halves), one on m << 16 (IMAD, FMA pipe: high half = min of the low
// halves) -- and one PRMT repacks them.  Per step of the pair: 15 ALU-pipe instructions (4 VIMNMX3, 4 VADD2, 4 VIADDMNMX,
// 2 min tree, 1 PRMT), 8 on the FMA pipe, 2 SHFL, 2 CREDUX; two sgm_step<2> take 24, ~8, 4 and 2.
__device__ __forceinline__ uint32_t sgm_step_pair(uint32_t (&O)[4], const uint32_t (&I)[4], uint32_t minI2,
                                                  const uint32_t (&Cv)[4], uint32_t p1x2, uint32_t k2, const SgmLane& s) {
    uint32_t Ip[4];
#pragma unroll
    for (int k = 0; k < 4; k++) Ip[k] = sgm_madlo(I[k], s.one, p1x2);
    const uint32_t up = sgm_madlo(__shfl_up_sync(0xffffffffu, Ip[3], 1), s.upm, s.upa);
    const uint32_t dn = sgm_madlo(__shfl_down_sync(0xffffffffu, Ip[0], 1), s.dnm, s.dna);
    const uint32_t nd2 = sgm_madlo(minI2, s.neg1, k2);
    uint32_t Ln[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const uint32_t t = __vimin3_u16x2(I[k], k ? Ip[k - 1] : up, k < 3 ? Ip[k + 1] : dn);
        Ln[k] = __viaddmin_u16x2(t, __vadd2(Cv[k], nd2), Cv[k]);
    }
    const uint32_t mn = __vimin3_u16x2(__vminu2(Ln[0], Ln[1]), Ln[2], Ln[3]);
#pragma unroll
    for (int k = 0; k < 4; k++) O[k] = Ln[k];
    const uint32_t hi = __reduce_min_sync(0xffffffffu, mn);
    const uint32_t lo = __reduce_min_sync(0xffffffffu, sgm_madlo(mn, s.m64k, s.zero));
    return __byte_perm(lo, hi, 0x7632);
}

}  // namespace l3d
