// Instruction-mix comparison of the SGM step forms (csrc/sgm_step.cuh) on one B200:
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/ubench/sgmstep tools/ubench/sgmstep.cu && tools/ubench/sgmstep
// Each warp runs NCH independent path recurrences (like the three previous-row paths of sgbm_vgroup_kernel) over the
// same shared-memory cost rows; 16 warps per CTA, one CTA per SM.  Prints cycles per (warp, step) and checks that all
// forms give identical bits.
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>
#include "../../laser_3d_reconstruction_b200/csrc/sgm_step.cuh"
using namespace l3d;

// round-1 form: literal zero operand, IADD3 for -(min + P2)
template <int NP>
__device__ __forceinline__ uint32_t step_lit0(uint32_t (&O)[NP], const uint32_t (&I)[NP], uint32_t minI2,
                                              const uint32_t (&Cv)[NP], uint32_t p1x2, uint32_t k2, uint32_t selA, uint32_t selB) {
    constexpr uint32_t INF = 0x7fff7fffu;
    const uint32_t up = __shfl_up_sync(0xffffffffu, I[NP - 1], 1);
    const uint32_t dn = __shfl_down_sync(0xffffffffu, I[0], 1);
    const uint32_t nd2 = k2 - minI2;
    const uint32_t pm2 = nd2 + p1x2;
    uint32_t mn = INF;
    uint32_t Ln[NP];
#pragma unroll
    for (int k = 0; k < NP; k++) {
        const uint32_t prev = k ? I[k - 1] : up;
        const uint32_t next = (k < NP - 1) ? I[k + 1] : dn;
        const uint32_t dm1 = k ? __byte_perm(prev, I[k], 0x5432) : __byte_perm(prev, I[k], selA);
        const uint32_t dp1 = (k < NP - 1) ? __byte_perm(I[k], next, 0x5432) : __byte_perm(I[k], next, selB);
        uint32_t t = __viaddmin_s16x2(I[k], nd2, 0u);
        t = __viaddmin_s16x2(dm1, pm2, t);
        t = __viaddmin_s16x2(dp1, pm2, t);
        Ln[k] = __vadd2(Cv[k], t);
        mn = __vminu2(mn, Ln[k]);
    }
#pragma unroll
    for (int k = 0; k < NP; k++) O[k] = Ln[k];
    mn = __vminu2(mn, __byte_perm(mn, mn, 0x1032));
    return __reduce_min_sync(0xffffffffu, mn);
}


// ---- round-2 experiments: move carry-free packed adds to the FMA pipe (IMAD with an opaque multiplier)
// FORM 3: I + P1 once per word (IMAD), neighbour words built from the sums, T = VIMNMX3(I, F[k], F[k+1])
// FORM 4: FORM 3 + L = min(T, delta) + (C - delta): one VIMNMX, two IMADs (32-bit modular arithmetic is exact because
//         the final halves lie in [0, 65535])
// FORM 5: FORM 4 + min tree as VIMNMX, CREDUX(hi), IMAD.SHL, CREDUX(lo), uniform min
template <int NP, int FORM>
__device__ __forceinline__ uint32_t step_fma(uint32_t (&O)[NP], const uint32_t (&I)[NP], uint32_t minI2,
                                             const uint32_t (&Cv)[NP], uint32_t p1x2, uint32_t k2, uint32_t p2x2,
                                             const SgmLane& s, uint32_t one) {
    uint32_t Ip[NP];
#pragma unroll
    for (int k = 0; k < NP; k++) Ip[k] = sgm_madlo(I[k], one, p1x2);
    const uint32_t up = __shfl_up_sync(0xffffffffu, Ip[NP - 1], 1);
    const uint32_t dn = __shfl_down_sync(0xffffffffu, Ip[0], 1);
    uint32_t F[NP + 1];
    F[0] = __byte_perm(up, Ip[0], s.selA);
    F[NP] = __byte_perm(Ip[NP - 1], dn, s.selB);
#pragma unroll
    for (int k = 1; k < NP; k++) F[k] = __byte_perm(Ip[k - 1], Ip[k], 0x5432);
    uint32_t Ln[NP];
    if (FORM == 9) {   // FORM 3 with L = min(T + (C - delta), C): no zero operand
        const uint32_t nd2 = sgm_madlo(minI2, s.neg1, k2);
#pragma unroll
        for (int k = 0; k < NP; k++) {
            const uint32_t t = __vimin3_u16x2(I[k], F[k], F[k + 1]);
            Ln[k] = __viaddmin_u16x2(t, __vadd2(Cv[k], nd2), Cv[k]);
        }
    } else if (FORM == 3) {
        const uint32_t nd2 = sgm_madlo(minI2, s.neg1, k2);
#pragma unroll
        for (int k = 0; k < NP; k++) {
            const uint32_t t = __vimin3_u16x2(I[k], F[k], F[k + 1]);
            Ln[k] = __vadd2(Cv[k], __viaddmin_s16x2(t, nd2, s.zero));
        }
    } else {
        const uint32_t delta2 = sgm_madlo(minI2, one, p2x2);
#pragma unroll
        for (int k = 0; k < NP; k++) {
            const uint32_t t = __vimin3_u16x2(I[k], F[k], F[k + 1]);
            const uint32_t u = __vminu2(t, delta2);
            const uint32_t cd = sgm_madlo(delta2, s.neg1, Cv[k]);
            Ln[k] = sgm_madlo(u, one, cd);
        }
    }
    uint32_t mn = Ln[0];
    if (NP == 2) mn = __vminu2(Ln[0], Ln[1]);
    if (NP == 4) mn = __vimin3_u16x2(__vminu2(Ln[0], Ln[1]), Ln[2], Ln[3]);
#pragma unroll
    for (int k = 0; k < NP; k++) O[k] = Ln[k];
    if (FORM == 5) {
        const uint32_t hi = __reduce_min_sync(0xffffffffu, mn);
        const uint32_t lo = __reduce_min_sync(0xffffffffu, sgm_madlo(mn, s.m64k, s.zero));
        const uint32_t m = min(hi, lo) >> 16;
        return m * 0x10001u;
    }
    mn = __vminu2(mn, __byte_perm(mn, mn, 0x1032));
    if (FORM == 6) return mn;  // timing only: no warp reduction (wrong bits)
    if (FORM == 7) {           // timing/bits: shuffle butterfly instead of CREDUX
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) mn = __vminu2(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        return mn;
    }
    if (FORM == 8) {           // non-coupled REDUX (result in a vector register)
        uint32_t r;
        asm volatile("redux.sync.min.u32 %0, %1, 0xffffffff;" : "=r"(r) : "r"(mn));
        return r;
    }
    return __reduce_min_sync(0xffffffffu, mn);
}

constexpr int ROWS = 64, NCH = 3;
template <int NP, int FORM>
__global__ void __launch_bounds__(512) bench(const uint32_t* __restrict__ cost, uint32_t* out, int iters, int P1, int P2,
                                             uint32_t zero, long long* cyc) {
    __shared__ uint32_t cs[ROWS][32 * NP];
    for (int i = threadIdx.x; i < ROWS * 32 * NP; i += blockDim.x) (&cs[0][0])[i] = cost[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const uint32_t p1x2 = (uint32_t)P1 * 0x10001u, k2 = (0x10000u - (uint32_t)P2) * 0x10001u;
    const uint32_t selA = lane == 0 ? 0x5454u : 0x5432u, selB = lane == 31 ? 0x3232u : 0x5432u;
    const SgmLane sl = sgm_lane_init(lane, zero);
    const uint32_t one = zero + 1u, p2x2 = (uint32_t)P2 * 0x10001u;
    uint32_t L[NCH][NP], mn[NCH];
    for (int c = 0; c < NCH; c++) { for (int k = 0; k < NP; k++) L[c][k] = 0; mn[c] = 0; }
    long long t0 = clock64();
    for (int it = 0; it < iters; it++) {
        const int r = it & (ROWS - 1);
        uint32_t Cw[NP];
#pragma unroll
        for (int c = 0; c < NCH; c++) {
#pragma unroll
            for (int k = 0; k < NP; k++) Cw[k] = cs[(r + c) & (ROWS - 1)][lane * NP + k];
            if (FORM == 0) mn[c] = step_lit0<NP>(L[c], L[c], mn[c], Cw, p1x2, k2, selA, selB);
            if (FORM == 1) mn[c] = sgm_step<NP, false>(L[c], L[c], mn[c], Cw, p1x2, k2, sl);
            if (FORM == 2) mn[c] = sgm_step<NP, true>(L[c], L[c], mn[c], Cw, p1x2, k2, sl);
            if (FORM >= 3) mn[c] = step_fma<NP, FORM>(L[c], L[c], mn[c], Cw, p1x2, k2, p2x2, sl, one);
        }
    }
    long long t1 = clock64();
    uint32_t acc = 0;
    for (int c = 0; c < NCH; c++) { for (int k = 0; k < NP; k++) acc = acc * 31u + L[c][k]; acc = acc * 31u + mn[c]; }
    out[blockIdx.x * blockDim.x + threadIdx.x] = acc;
    if (threadIdx.x == 0 && blockIdx.x == 0) *cyc = t1 - t0;
}

// The paired form (sgm_step_pair) against sgm_step<2> on the same work: NPAIR pairs of D = 128 recurrences per warp,
// pair c = recurrences (2c, 2c + 1) over cost rows (r, r + 1), each pair starting from its own state (so that nothing is
// common to two pairs).  PAIRED = false runs the 2 NPAIR recurrences one by one with sgm_step<2>; PAIRED = true
// interleaves the two cost rows once per step (four PRMTs, shared by the pairs, as in the kernel where the A, V and B
// paths of a column pair read the same costs) and runs sgm_step_pair.  Both hash the states in sgm_step's layout.
constexpr int NPAIR = 3;
template <bool PAIRED>
__global__ void __launch_bounds__(512) bench_pair(const uint32_t* __restrict__ cost, uint32_t* out, int iters, int P1, int P2,
                                                  uint32_t zero, long long* cyc) {
    __shared__ uint32_t cs[ROWS][64];
    for (int i = threadIdx.x; i < ROWS * 64; i += blockDim.x) (&cs[0][0])[i] = cost[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const uint32_t p1x2 = (uint32_t)P1 * 0x10001u, k2 = (0x10000u - (uint32_t)P2) * 0x10001u;
    const SgmLane sl = sgm_lane_init(lane, zero);
    uint32_t L[2 * NPAIR][2], mn[2 * NPAIR];   // sgm_step's layout (PAIRED = false)
    uint32_t P[NPAIR][4], pm[NPAIR];           // paired layout
    for (int c = 0; c < NPAIR; c++) {
        const uint32_t v = (uint32_t)(100 * c + 7) * 0x10001u;
        for (int k = 0; k < 2; k++) L[2 * c][k] = L[2 * c + 1][k] = v;
        for (int k = 0; k < 4; k++) P[c][k] = v;
        mn[2 * c] = mn[2 * c + 1] = v; pm[c] = v;
    }
    long long t0 = clock64();
    for (int it = 0; it < iters; it++) {
        const int r = it & (ROWS - 1);
        const uint2 ca = *(const uint2*)&cs[r][lane * 2], cb = *(const uint2*)&cs[(r + 1) & (ROWS - 1)][lane * 2];
        if (PAIRED) {
            const uint32_t Cw[4] = {__byte_perm(ca.x, cb.x, 0x5410), __byte_perm(ca.x, cb.x, 0x7632),
                                    __byte_perm(ca.y, cb.y, 0x5410), __byte_perm(ca.y, cb.y, 0x7632)};
#pragma unroll
            for (int c = 0; c < NPAIR; c++) pm[c] = sgm_step_pair(P[c], P[c], pm[c], Cw, p1x2, k2, sl);
        } else {
            const uint32_t Ca[2] = {ca.x, ca.y}, Cb[2] = {cb.x, cb.y};
#pragma unroll
            for (int c = 0; c < NPAIR; c++) {
                mn[2 * c] = sgm_step<2>(L[2 * c], L[2 * c], mn[2 * c], Ca, p1x2, k2, sl);
                mn[2 * c + 1] = sgm_step<2>(L[2 * c + 1], L[2 * c + 1], mn[2 * c + 1], Cb, p1x2, k2, sl);
            }
        }
    }
    long long t1 = clock64();
    if (PAIRED) {
        for (int c = 0; c < NPAIR; c++) {
            L[2 * c][0] = __byte_perm(P[c][0], P[c][1], 0x5410); L[2 * c][1] = __byte_perm(P[c][2], P[c][3], 0x5410);
            L[2 * c + 1][0] = __byte_perm(P[c][0], P[c][1], 0x7632); L[2 * c + 1][1] = __byte_perm(P[c][2], P[c][3], 0x7632);
            mn[2 * c] = (pm[c] & 0xffffu) * 0x10001u; mn[2 * c + 1] = (pm[c] >> 16) * 0x10001u;
        }
    }
    uint32_t acc = 0;
    for (int c = 0; c < 2 * NPAIR; c++) { for (int k = 0; k < 2; k++) acc = acc * 31u + L[c][k]; acc = acc * 31u + mn[c]; }
    out[blockIdx.x * blockDim.x + threadIdx.x] = acc;
    if (threadIdx.x == 0 && blockIdx.x == 0) *cyc = t1 - t0;
}

template <bool PAIRED>
static void run_pair(const char* name, const uint32_t* cost, uint32_t* out, uint32_t* host, long long* cyc, int P1, int P2) {
    const int iters = 20000, n = 148 * 512;
    cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
    bench_pair<PAIRED><<<148, 512>>>(cost, out, 100, P1, P2, 0u, cyc);
    cudaEventRecord(a);
    bench_pair<PAIRED><<<148, 512>>>(cost, out, iters, P1, P2, 0u, cyc);
    cudaEventRecord(b); cudaEventSynchronize(b);
    float ms; cudaEventElapsedTime(&ms, a, b);
    long long c; cudaMemcpy(&c, cyc, 8, cudaMemcpyDeviceToHost);
    cudaMemcpy(host, out, n * 4, cudaMemcpyDeviceToHost);
    unsigned long long h = 0; for (int i = 0; i < n; i++) h = h * 1000003ull + host[i];
    const double per = (double)c / (iters * 2 * NPAIR);
    printf("D=128 %-34s %8.3f ms  %7.2f cycles per (warp, vector-step) at 16 warps/SM = %6.2f per SM-subpartition-step   hash %016llx  err=%s\n",
           name, ms, per, per / 4.0, h, cudaGetErrorString(cudaGetLastError()));
}

template <int NP, int FORM>
static void run(const char* name, const uint32_t* cost, uint32_t* out, uint32_t* host, long long* cyc, int P1, int P2) {
    const int iters = 20000, n = 148 * 512;
    cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
    bench<NP, FORM><<<148, 512>>>(cost, out, 100, P1, P2, 0u, cyc);
    cudaEventRecord(a);
    bench<NP, FORM><<<148, 512>>>(cost, out, iters, P1, P2, 0u, cyc);
    cudaEventRecord(b); cudaEventSynchronize(b);
    float ms; cudaEventElapsedTime(&ms, a, b);
    long long c; cudaMemcpy(&c, cyc, 8, cudaMemcpyDeviceToHost);
    cudaMemcpy(host, out, n * 4, cudaMemcpyDeviceToHost);
    unsigned long long h = 0; for (int i = 0; i < n; i++) h = h * 1000003ull + host[i];
    printf("NP=%d %-28s %8.3f ms  %7.2f cycles per (warp, step) at 16 warps/SM = %6.2f per SM-subpartition-step   hash %016llx  err=%s\n",
           NP, name, ms, (double)c / (iters * NCH), (double)c / (iters * NCH) / 4.0, h, cudaGetErrorString(cudaGetLastError()));
}

int main() {
    const int P1 = 1944, P2 = 7776;
    uint32_t *cost, *out; long long* cyc;
    const int ncost = ROWS * 32 * 4;
    uint32_t* hc = new uint32_t[ncost];
    uint32_t s = 12345;
    for (int i = 0; i < ncost; i++) {  // C in [P2, P2 + 15000]: both halves
        s = s * 1664525u + 1013904223u; uint32_t a = P2 + (s >> 8) % 15000;
        s = s * 1664525u + 1013904223u; uint32_t b = P2 + (s >> 8) % 15000;
        hc[i] = a | (b << 16);
    }
    cudaMalloc(&cost, ncost * 4); cudaMalloc(&out, 148 * 512 * 4); cudaMalloc(&cyc, 8);
    cudaMemcpy(cost, hc, ncost * 4, cudaMemcpyHostToDevice);
    uint32_t* host = new uint32_t[148 * 512];
    run<2, 0>("alu, literal 0 (round 1)", cost, out, host, cyc, P1, P2);
    run<2, 1>("register 0, delta last", cost, out, host, cyc, P1, P2);
    run<2, 2>("delta last + FMA funnels", cost, out, host, cyc, P1, P2);
    run<2, 3>("I+P1 by IMAD, VIMNMX3", cost, out, host, cyc, P1, P2);
    run<2, 4>("+ L = min(T,delta) + (C-delta)", cost, out, host, cyc, P1, P2);
    run<2, 5>("+ two CREDUX min tree", cost, out, host, cyc, P1, P2);
    run<2, 9>("form 3, min(T + (C-delta), C)", cost, out, host, cyc, P1, P2);
    run_pair<false>("sgm_step<2>, 6 recurrences", cost, out, host, cyc, P1, P2);
    run_pair<true>("sgm_step_pair, 3 pairs", cost, out, host, cyc, P1, P2);
    run_pair<false>("sgm_step<2>, 6 recurrences", cost, out, host, cyc, P1, P2);
    run_pair<true>("sgm_step_pair, 3 pairs", cost, out, host, cyc, P1, P2);
    run<4, 9>("form 3, min(T + (C-delta), C)", cost, out, host, cyc, P1, P2);
    run<1, 9>("form 3, min(T + (C-delta), C)", cost, out, host, cyc, P1, P2);
    run<2, 6>("form 4 without the reduction", cost, out, host, cyc, P1, P2);
    run<2, 7>("form 4, shuffle butterfly", cost, out, host, cyc, P1, P2);
    run<2, 8>("form 4, redux.sync asm", cost, out, host, cyc, P1, P2);
    run<4, 0>("alu, literal 0 (round 1)", cost, out, host, cyc, P1, P2);
    run<4, 1>("register 0, delta last", cost, out, host, cyc, P1, P2);
    run<4, 2>("delta last + FMA funnels", cost, out, host, cyc, P1, P2);
    run<4, 3>("I+P1 by IMAD, VIMNMX3", cost, out, host, cyc, P1, P2);
    run<4, 4>("+ L = min(T,delta) + (C-delta)", cost, out, host, cyc, P1, P2);
    run<4, 5>("+ two CREDUX min tree", cost, out, host, cyc, P1, P2);
    run<1, 0>("alu, literal 0 (round 1)", cost, out, host, cyc, P1, P2);
    run<1, 2>("delta last + FMA funnels", cost, out, host, cyc, P1, P2);
    run<1, 3>("I+P1 by IMAD, VIMNMX3", cost, out, host, cyc, P1, P2);
    run<1, 4>("+ L = min(T,delta) + (C-delta)", cost, out, host, cyc, P1, P2);
    run<1, 5>("+ two CREDUX min tree", cost, out, host, cyc, P1, P2);
    return 0;
}
