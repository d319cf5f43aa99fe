// planefit.cu -- the laser plane from a stereo-triangulated point cloud (include/l3d.h: l3d_fit_plane, DESIGN.md 4f):
// RANSAC over hypothesis planes through point triples, then least-squares refits on the inlier set.
//   RANSAC      every hypothesis's plane and its inlier count follow an exact f64 contract (round-to-nearest, no FMA,
//               fixed operation order) and the counts are integers, so any kernel layout -- and the numpy restatement
//               in oracle/plane_fit.py -- picks the same winner
//   refinement  centroid and centred covariance of the inlier set as per-CTA partials over a layout fixed by n, summed
//               on the host in CTA order (identical bits from run to run); the 3x3 eigenproblem by Jacobi on the host
#include <algorithm>
#include <cmath>

#include "common.cuh"

namespace l3d {

constexpr int PF_THREADS = 128;             // scoring CTA: one thread per PF_HPT hypotheses
constexpr int PF_HPT = 2;                   // hypotheses per thread: each point read from shared memory feeds two planes
constexpr int PF_TILE = 1024;               // points staged in shared memory per step (24 KB)
constexpr int PF_RED_THREADS = 256;
constexpr int PF_RED_BLOCKS = 4 * NUM_SMS;  // reduction CTAs for large n; the partials layout depends on n alone
constexpr int PF_MAX_FITS = 10;

__device__ __forceinline__ unsigned long long pf_point_index(unsigned long long seed, unsigned long long j, int n) {
    unsigned long long z = seed + j * 0x9E3779B97F4A7C15ull;  // j = 3h + k + 1, mod 2^64
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    return z % (unsigned long long)n;
}

__device__ __forceinline__ double pf_residual(double nx, double ny, double nz, double d, double x, double y, double z) {
    return __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(nx, x), __dmul_rn(ny, y)), __dmul_rn(nz, z)), d);
}

// one thread per hypothesis: its plane (NaN for an invalid one, which then counts no inlier) and its count's start value
// (0, or -1 for an invalid hypothesis, so that it never wins)
__global__ void pf_planes_kernel(const double* __restrict__ pts, int n, int hyps, unsigned long long seed,
                                 double4* __restrict__ planes, int* __restrict__ count) {
    const int h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= hyps) return;
    double p[3][3];
    bool ok = true;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const unsigned long long i = pf_point_index(seed, 3ull * (unsigned long long)h + k + 1, n);
#pragma unroll
        for (int a = 0; a < 3; a++) { p[k][a] = pts[i * 3 + a]; ok = ok && isfinite(p[k][a]); }
    }
    const double ux = __dsub_rn(p[1][0], p[0][0]), uy = __dsub_rn(p[1][1], p[0][1]), uz = __dsub_rn(p[1][2], p[0][2]);
    const double vx = __dsub_rn(p[2][0], p[0][0]), vy = __dsub_rn(p[2][1], p[0][1]), vz = __dsub_rn(p[2][2], p[0][2]);
    double nx = __dsub_rn(__dmul_rn(uy, vz), __dmul_rn(uz, vy));
    double ny = __dsub_rn(__dmul_rn(uz, vx), __dmul_rn(ux, vz));
    double nz = __dsub_rn(__dmul_rn(ux, vy), __dmul_rn(uy, vx));
    const double s = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(nx, nx), __dmul_rn(ny, ny)), __dmul_rn(nz, nz)));
    if (!(ok && s > 0.0 && s < __longlong_as_double(0x7ff0000000000000ll))) {
        const double nan = __longlong_as_double(0x7ff8000000000000ll);
        planes[h] = make_double4(nan, nan, nan, nan);
        count[h] = -1;
        return;
    }
    nx = __ddiv_rn(nx, s); ny = __ddiv_rn(ny, s); nz = __ddiv_rn(nz, s);
    const double d = -__dadd_rn(__dadd_rn(__dmul_rn(nx, p[0][0]), __dmul_rn(ny, p[0][1])), __dmul_rn(nz, p[0][2]));
    planes[h] = make_double4(nx, ny, nz, d);
    count[h] = 0;
}

// grid (hypothesis groups, point ranges): each thread keeps PF_HPT planes in registers and sweeps its CTA's point range in
// shared-memory tiles (every thread reads the same point: a broadcast); one integer atomicAdd per hypothesis and CTA
__global__ void __launch_bounds__(PF_THREADS) pf_score_kernel(const double* __restrict__ pts, int n, int hyps,
                                                              const double4* __restrict__ planes, double thr,
                                                              int tiles_per_cta, int* __restrict__ count) {
    __shared__ double2 sxy[PF_TILE];
    __shared__ double sz[PF_TILE];
    const int h0 = (blockIdx.x * PF_THREADS + threadIdx.x) * PF_HPT;
    double4 pl[PF_HPT];
    int c[PF_HPT];
#pragma unroll
    for (int j = 0; j < PF_HPT; j++) {
        const double nan = __longlong_as_double(0x7ff8000000000000ll);
        pl[j] = h0 + j < hyps ? planes[h0 + j] : make_double4(nan, nan, nan, nan);
        c[j] = 0;
    }
    const long long begin = (long long)blockIdx.y * tiles_per_cta * PF_TILE;
    const long long end = min((long long)n, begin + (long long)tiles_per_cta * PF_TILE);
    for (long long t0 = begin; t0 < end; t0 += PF_TILE) {
        const int tn = (int)min((long long)PF_TILE, end - t0);
        __syncthreads();
        for (int q = threadIdx.x; q < tn; q += PF_THREADS) {
            const double* s = pts + (size_t)(t0 + q) * 3;
            sxy[q] = make_double2(s[0], s[1]);
            sz[q] = s[2];
        }
        __syncthreads();
#pragma unroll 4
        for (int q = 0; q < tn; q++) {
            const double2 xy = sxy[q];
            const double z = sz[q];
#pragma unroll
            for (int j = 0; j < PF_HPT; j++)
                c[j] += fabs(pf_residual(pl[j].x, pl[j].y, pl[j].z, pl[j].w, xy.x, xy.y, z)) <= thr;  // NaN: never
        }
    }
#pragma unroll
    for (int j = 0; j < PF_HPT; j++)
        if (h0 + j < hyps && c[j]) atomicAdd(count + h0 + j, c[j]);
}

// CTA b covers points [b * chunk, (b + 1) * chunk); thread t its points t, t + PF_RED_THREADS, ...; then a fixed tree
template <int K>
__device__ __forceinline__ void pf_block_sum(double (&acc)[K], double* __restrict__ out) {
    __shared__ double red[K][PF_RED_THREADS];
    const int t = threadIdx.x;
#pragma unroll
    for (int k = 0; k < K; k++) red[k][t] = acc[k];
    __syncthreads();
    for (int s = PF_RED_THREADS / 2; s > 0; s >>= 1) {
        if (t < s)
#pragma unroll
            for (int k = 0; k < K; k++) red[k][t] = __dadd_rn(red[k][t], red[k][t + s]);
        __syncthreads();
    }
    if (t < K) out[t] = red[t][0];
}

// centred == 0: per-CTA sums of x, y, z over the points in `mask`; centred != 0: of the six products of p - c
__global__ void __launch_bounds__(PF_RED_THREADS) pf_moments_kernel(const double* __restrict__ pts, int n, int chunk,
                                                                    const uint8_t* __restrict__ mask, int centred,
                                                                    double cx, double cy, double cz,
                                                                    double* __restrict__ partial) {
    double acc[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    const long long b0 = (long long)blockIdx.x * chunk, b1 = min((long long)n, b0 + chunk);
    for (long long i = b0 + threadIdx.x; i < b1; i += PF_RED_THREADS) {
        if (!mask[i]) continue;
        const double x = pts[i * 3], y = pts[i * 3 + 1], z = pts[i * 3 + 2];
        if (!centred) {
            acc[0] = __dadd_rn(acc[0], x); acc[1] = __dadd_rn(acc[1], y); acc[2] = __dadd_rn(acc[2], z);
        } else {
            const double dx = __dsub_rn(x, cx), dy = __dsub_rn(y, cy), dz = __dsub_rn(z, cz);
            acc[0] = __dadd_rn(acc[0], __dmul_rn(dx, dx)); acc[1] = __dadd_rn(acc[1], __dmul_rn(dx, dy));
            acc[2] = __dadd_rn(acc[2], __dmul_rn(dx, dz)); acc[3] = __dadd_rn(acc[3], __dmul_rn(dy, dy));
            acc[4] = __dadd_rn(acc[4], __dmul_rn(dy, dz)); acc[5] = __dadd_rn(acc[5], __dmul_rn(dz, dz));
        }
    }
    pf_block_sum<6>(acc, partial + (size_t)blockIdx.x * 6);
}

// the inlier set of a plane (the RANSAC residual, bit for bit): mask, counters[0] += inliers, counters[1] += points whose
// membership differs from `prev` (may be null), per-CTA sums of the inliers' squared residuals
__global__ void __launch_bounds__(PF_RED_THREADS) pf_select_kernel(const double* __restrict__ pts, int n, int chunk,
                                                                   double nx, double ny, double nz, double d, double thr,
                                                                   const uint8_t* __restrict__ prev,
                                                                   uint8_t* __restrict__ mask, int* __restrict__ counters,
                                                                   double* __restrict__ partial_r2) {
    __shared__ int s_in, s_changed;
    if (threadIdx.x == 0) { s_in = 0; s_changed = 0; }
    __syncthreads();
    double acc[1] = {0.0};
    int in = 0, changed = 0;
    const long long b0 = (long long)blockIdx.x * chunk, b1 = min((long long)n, b0 + chunk);
    for (long long i = b0 + threadIdx.x; i < b1; i += PF_RED_THREADS) {
        const double r = pf_residual(nx, ny, nz, d, pts[i * 3], pts[i * 3 + 1], pts[i * 3 + 2]);
        const uint8_t m = fabs(r) <= thr;
        mask[i] = m;
        if (m) { in++; acc[0] = __dadd_rn(acc[0], __dmul_rn(r, r)); }
        if (prev && prev[i] != m) changed++;
    }
    if (in) atomicAdd(&s_in, in);
    if (changed) atomicAdd(&s_changed, changed);
    pf_block_sum<1>(acc, partial_r2 + blockIdx.x);  // its __syncthreads orders the shared counters too
    if (threadIdx.x == 0) {
        if (s_in) atomicAdd(counters, s_in);
        if (s_changed) atomicAdd(counters + 1, s_changed);
    }
}

// cyclic Jacobi on a symmetric 3x3 matrix (row-major): w ascending, column k of V (row-major) the unit eigenvector of w[k]
static void jacobi3(const double A[9], double w[3], double V[9]) {
    double a[3][3], v[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
    double scale = 0.0;
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) { a[i][j] = A[i * 3 + j]; scale = std::max(scale, std::fabs(a[i][j])); }
    static const int P[3][2] = {{0, 1}, {0, 2}, {1, 2}};
    for (int sweep = 0; sweep < 64; sweep++) {
        bool rotated = false;
        for (const auto& pq : P) {
            const int p = pq[0], q = pq[1];
            if (std::fabs(a[p][q]) <= 1e-300 + 1e-22 * scale) continue;
            rotated = true;
            const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
            const double t = (theta >= 0.0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
            const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
            for (int k = 0; k < 3; k++) {
                const double akp = a[k][p], akq = a[k][q];
                a[k][p] = c * akp - s * akq; a[k][q] = s * akp + c * akq;
            }
            for (int k = 0; k < 3; k++) {
                const double apk = a[p][k], aqk = a[q][k];
                a[p][k] = c * apk - s * aqk; a[q][k] = s * apk + c * aqk;
            }
            for (int k = 0; k < 3; k++) {
                const double vkp = v[k][p], vkq = v[k][q];
                v[k][p] = c * vkp - s * vkq; v[k][q] = s * vkp + c * vkq;
            }
        }
        if (!rotated) break;
    }
    int order[3] = {0, 1, 2};
    std::sort(order, order + 3, [&](int x, int y) { return a[x][x] < a[y][y]; });
    for (int k = 0; k < 3; k++) {
        w[k] = a[order[k]][order[k]];
        for (int i = 0; i < 3; i++) V[i * 3 + k] = v[i][order[k]];
    }
}

// pts: device, n x 3 f64; arguments already checked by the caller.  *mask_dev = the result's inlier mask (device, n bytes)
int dev_fit_plane(Lane& L, const double* pts, int n, const l3d_plane_fit_params& prm, l3d_plane_fit_result* res,
                  const uint8_t** mask_dev) {
    const int hyps = prm.hypotheses;
    const double thr = prm.threshold;
    double4* planes = L.get<double4>(S_IO_A, hyps);
    int* count = L.get<int>(S_IO_B, hyps);
    uint8_t* masks = L.get<uint8_t>(S_IO_C, (size_t)2 * n);
    const int rblocks = std::min(PF_RED_BLOCKS, cdiv(n, PF_RED_THREADS));
    const int chunk = cdiv(n, rblocks);
    double* partial = L.get<double>(S_IO_D, (size_t)rblocks * 7);  // 6 moments + 1 squared-residual sum per CTA
    double* partial_r2 = partial + (size_t)rblocks * 6;
    int* counters = L.get<int>(S_IO_E, 2);

    // RANSAC
    L3D_LAUNCH(L, pf_planes_kernel, cdiv(hyps, 128), 128, 0, pts, n, hyps, (unsigned long long)prm.seed, planes, count);
    const int gx = cdiv(hyps, PF_THREADS * PF_HPT);
    const int tiles = cdiv(n, PF_TILE);
    int gy = std::min(tiles, std::max(1, cdiv(8 * NUM_SMS, gx)));
    const int tiles_per_cta = cdiv(tiles, gy);
    gy = cdiv(tiles, tiles_per_cta);
    L3D_LAUNCH(L, pf_score_kernel, dim3(gx, gy), PF_THREADS, 0, pts, n, hyps, planes, thr, tiles_per_cta, count);
    std::vector<int> hc(hyps);
    L3D_CHECK(L, cudaMemcpyAsync(hc.data(), count, sizeof(int) * hyps, cudaMemcpyDeviceToHost, L.stream));
    L3D_CHECK(L, cudaStreamSynchronize(L.stream));
    const int win = (int)(std::max_element(hc.begin(), hc.end()) - hc.begin());  // the first maximum: lowest h
    if (hc[win] < 0) { set_err(L.err, "invalid argument: plane fit: no hypothesis has three finite, non-collinear points"); return L3D_ERR_ARG; }
    res->hypothesis = win;
    res->hypothesis_inliers = hc[win];
    double4 wp;
    L3D_CHECK(L, cudaMemcpyAsync(&wp, planes + win, sizeof(double4), cudaMemcpyDeviceToHost, L.stream));
    L3D_CHECK(L, cudaStreamSynchronize(L.stream));

    // the inlier set S of a plane -> counters {|S|, |S xor prev|}, its squared residual sum
    std::vector<double> hp((size_t)rblocks * 6);
    auto select = [&](const double* pl, const uint8_t* prev, uint8_t* out, int* in, int* changed, double* r2) -> int {
        L3D_CHECK(L, cudaMemsetAsync(counters, 0, sizeof(int) * 2, L.stream));
        L3D_LAUNCH(L, pf_select_kernel, rblocks, PF_RED_THREADS, 0, pts, n, chunk, pl[0], pl[1], pl[2], pl[3], thr, prev, out,
                   counters, partial_r2);
        int hcnt[2];
        L3D_CHECK(L, cudaMemcpyAsync(hcnt, counters, sizeof(hcnt), cudaMemcpyDeviceToHost, L.stream));
        L3D_CHECK(L, cudaMemcpyAsync(hp.data(), partial_r2, sizeof(double) * rblocks, cudaMemcpyDeviceToHost, L.stream));
        L3D_CHECK(L, cudaStreamSynchronize(L.stream));
        *in = hcnt[0];
        *changed = hcnt[1];
        double s = 0.0;
        for (int b = 0; b < rblocks; b++) s += hp[b];
        *r2 = s;
        return L3D_OK;
    };
    // per-CTA moments summed in CTA order
    auto moments = [&](const uint8_t* m, int centred, const double* c, double* sums) -> int {
        L3D_LAUNCH(L, pf_moments_kernel, rblocks, PF_RED_THREADS, 0, pts, n, chunk, m, centred, c[0], c[1], c[2], partial);
        L3D_CHECK(L, cudaMemcpyAsync(hp.data(), partial, sizeof(double) * rblocks * 6, cudaMemcpyDeviceToHost, L.stream));
        L3D_CHECK(L, cudaStreamSynchronize(L.stream));
        for (int k = 0; k < 6; k++) sums[k] = 0.0;
        for (int b = 0; b < rblocks; b++)
            for (int k = 0; k < 6; k++) sums[k] += hp[(size_t)b * 6 + k];
        return L3D_OK;
    };

    uint8_t* S = masks;
    uint8_t* S2 = masks + n;
    int m = 0, changed = 0;
    double r2 = 0.0;
    const double wpl[4] = {wp.x, wp.y, wp.z, wp.w};
    int rc = select(wpl, nullptr, S, &m, &changed, &r2);
    if (rc != L3D_OK) return rc;
    double plane[4] = {0, 0, 0, 0}, w[3] = {0, 0, 0};
    int fits = 0;
    for (;;) {
        if (m < 3) { set_err(L.err, "invalid argument: plane fit: %d inlier(s) left, a plane needs 3", m); return L3D_ERR_ARG; }
        const double zero[3] = {0, 0, 0};
        double sum[6], cov[6];
        if ((rc = moments(S, 0, zero, sum)) != L3D_OK) return rc;
        const double c[3] = {sum[0] / m, sum[1] / m, sum[2] / m};
        if ((rc = moments(S, 1, c, cov)) != L3D_OK) return rc;
        const double A[9] = {cov[0] / m, cov[1] / m, cov[2] / m, cov[1] / m, cov[3] / m, cov[4] / m, cov[2] / m, cov[4] / m, cov[5] / m};
        double V[9];
        jacobi3(A, w, V);
        plane[0] = V[0]; plane[1] = V[3]; plane[2] = V[6];
        plane[3] = -((plane[0] * c[0] + plane[1] * c[1]) + plane[2] * c[2]);
        int m2 = 0;
        if ((rc = select(plane, S, S2, &m2, &changed, &r2)) != L3D_OK) return rc;
        fits++;
        std::swap(S, S2);
        m = m2;
        if (changed == 0 || fits == PF_MAX_FITS) break;
    }
    if (m < 3) { set_err(L.err, "invalid argument: plane fit: %d inlier(s) left, a plane needs 3", m); return L3D_ERR_ARG; }
    const double sgn = plane[3] < 0.0 ? -1.0 : 1.0;
    for (int k = 0; k < 4; k++) res->plane[k] = sgn * plane[k];
    for (int k = 0; k < 3; k++) res->eig[k] = w[k];
    res->inliers = m;
    res->rms = std::sqrt(r2 / m);
    res->refits = fits;
    *mask_dev = S;
    return L3D_OK;
}

}  // namespace l3d
