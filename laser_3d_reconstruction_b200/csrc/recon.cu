// recon.cu -- K5b: laser pixel -> 3D point.
//   PLANE            Reconstructor.reconstruct_point/_refraction_correction/reconstruct_laser_line
//                    core/reconstruction.py:30-143  (f64; the refraction sign quirk is preserved)
//   DEPTH            Reconstructor.reconstruct_from_depth  core/reconstruction.py:145-182
//                    (z = depth/1000 is the reference's unit bug, preserved; f32 divide as numpy 2
//                    evaluates np.float32 / python-float)
//   DISPARITY        ImprovedLaserReconstructor.reconstruct_from_disparity  improved_reconstruction.py:37-86
//   DISPARITY_MEDIAN .reconstruct_with_interpolation  improved_reconstruction.py:88-152
// One thread per point, then an order-preserving compaction (invalid points are dropped).
#include "common.cuh"

namespace l3d {

__global__ void row_scan_kernel(const int* __restrict__ cnt, int H, int* __restrict__ off, int* __restrict__ n);

struct ReconArgs {
    l3d_recon_params p;
    double Kinv[9];
};

__device__ __forceinline__ bool finite3(double a, double b, double c) { return isfinite(a) && isfinite(b) && isfinite(c); }
__device__ __forceinline__ bool notnan3(double a, double b, double c) { return !(isnan(a) || isnan(b) || isnan(c)); }

__device__ bool recon_plane(const ReconArgs& a, double u, double v, double* o) {
    const double* K = a.Kinv;
    double r0 = K[0] * u + K[1] * v + K[2], r1 = K[3] * u + K[4] * v + K[5], r2 = K[6] * u + K[7] * v + K[8];
    double nr = sqrt(r0 * r0 + r1 * r1 + r2 * r2);
    r0 /= nr; r1 /= nr; r2 /= nr;
    const double pa = a.p.plane[0], pb = a.p.plane[1], pc = a.p.plane[2], pd = a.p.plane[3];
    double den = pa * r0 + pb * r1 + pc * r2;
    if (fabs(den) < 1e-10) return false;
    double t = -pd / den;
    if (t < 0) return false;
    double p0 = t * r0, p1 = t * r1, p2 = t * r2;
    if (a.p.use_refraction) {
        const double k = 1.0 / a.p.n_water;
        double cos1 = -r2;  // -dot(ray, [0,0,1]): negative for forward rays, as in the reference
        double sin1 = sqrt(1 - cos1 * cos1);
        double sin2 = k * sin1;
        if (!(sin2 > 1)) {
            double cos2 = sqrt(1 - sin2 * sin2);
            double q0 = k * r0, q1 = k * r1, q2 = k * r2 + (k * cos1 - cos2);
            double nq = sqrt(q0 * q0 + q1 * q1 + q2 * q2);
            q0 /= nq; q1 /= nq; q2 /= nq;
            double den2 = pa * q0 + pb * q1 + pc * q2;
            if (!(fabs(den2) < 1e-10)) {
                double t2 = -pd / den2;  // no t<0 test on the refracted ray (reference behaviour)
                p0 = t2 * q0; p1 = t2 * q1; p2 = t2 * q2;
            }
        }
    }
    o[0] = p0; o[1] = p1; o[2] = p2;
    return notnan3(p0, p1, p2);
}

__device__ bool recon_depth(const ReconArgs& a, double u, double v, const float* img, int W, int H, double* o) {
    if (!(fabs(u) < 2147483647.0 && fabs(v) < 2147483647.0)) return false;
    int iu = (int)u, iv = (int)v;  // python int(): truncation toward zero
    if (!(0 <= iu && iu < W && 0 <= iv && iv < H)) return false;
    float depth = img[(size_t)iv * W + iu];
    if (!(depth > 0.f)) return false;
    double z = (double)__fdiv_rn(depth, 1000.0f);
    const double fx = a.p.K[0], fy = a.p.K[4], cx = a.p.K[2], cy = a.p.K[5];
    o[0] = __ddiv_rn(__dmul_rn(u - cx, z), fx);
    o[1] = __ddiv_rn(__dmul_rn(v - cy, z), fy);
    o[2] = z;
    return true;
}

// A disparity element as the reference sees it: the f32 map as is, or the matcher's int16 x16 disparity as
// `disp.astype(np.float32) / 16.0` (int16 -> f32 is exact and so is the power-of-two scale, |v| <= 32767).
__device__ __forceinline__ float disp_px(float v) { return v; }
__device__ __forceinline__ float disp_px(int16_t v) { return (float)v * 0.0625f; }

template <typename T>
__device__ bool recon_disp(const ReconArgs& a, double x, double y, const T* img, int W, int H, double* o) {
    if (!(fabs(x) < 2147483647.0 && fabs(y) < 2147483647.0)) return false;
    int px = (int)rint(x), py = (int)rint(y);  // python round(): half to even
    float disp;
    const float mind = (float)a.p.min_disparity;
    if (a.p.kind == L3D_RECON_DISPARITY) {
        if (px < 0 || px >= W || py < 0 || py >= H) return false;
        disp = disp_px(img[(size_t)py * W + px]);
        if (disp < mind || isnan(disp) || isinf(disp)) return false;
    } else {
        const int hw = a.p.window / 2;
        if (px < hw || px >= W - hw || py < hw || py >= H - hw) return false;
        // sorted by the raw element: the conversion is monotonic, so only the middle one(s) need converting
        T vals[81];
        int n = 0;
        for (int dy = -hw; dy <= hw; dy++)
            for (int dx = -hw; dx <= hw; dx++) {
                T k = img[(size_t)(py + dy) * W + px + dx];
                float d = disp_px(k);
                if (d >= mind && !isnan(d) && !isinf(d)) {
                    int j = n++;
                    while (j > 0 && vals[j - 1] > k) { vals[j] = vals[j - 1]; j--; }
                    vals[j] = k;
                }
            }
        if (n == 0) return false;
        // np.median on float32: odd -> middle, even -> f32 mean of the two middle values
        disp = (n & 1) ? disp_px(vals[n / 2]) : __fmul_rn(__fadd_rn(disp_px(vals[n / 2 - 1]), disp_px(vals[n / 2])), 0.5f);
    }
    double Z = __ddiv_rn(__dmul_rn(a.p.fx, a.p.baseline), (double)disp);
    double X = __ddiv_rn(__dmul_rn((double)px - a.p.cx, Z), a.p.fx);
    double Y = __ddiv_rn(__dmul_rn((double)py - a.p.cy, Z), a.p.fx);  // fx for Y too, as in the reference
    if (!(Z > 0 && Z < 10.0)) return false;
    o[0] = X; o[1] = Y; o[2] = Z;
    return true;
}

// T = float: l3d_reconstruct's host maps (every kind); T = int16_t: the frame pipeline's x16 disparity (DISPARITY kinds)
template <typename T>
__global__ void recon_points_kernel(ReconArgs a, const double* __restrict__ xy, const float* __restrict__ xyf,
                                    const int* __restrict__ n_dev, int n_max, const T* __restrict__ img, int W,
                                    int H, double* __restrict__ tmp, int* __restrict__ flag) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_max) return;
    int n = n_dev ? min(*n_dev, n_max) : n_max;
    bool ok = false;
    double o[3] = {0, 0, 0};
    if (i < n) {
        double u = xy ? xy[2 * i] : (double)xyf[2 * i], v = xy ? xy[2 * i + 1] : (double)xyf[2 * i + 1];
        if constexpr (std::is_same<T, int16_t>::value) ok = recon_disp(a, u, v, img, W, H, o);
        else if (a.p.kind == L3D_RECON_PLANE) ok = recon_plane(a, u, v, o);
        else if (a.p.kind == L3D_RECON_DEPTH) ok = recon_depth(a, u, v, img, W, H, o);
        else ok = recon_disp(a, u, v, img, W, H, o);
    }
    flag[i] = ok ? 1 : 0;
    tmp[3 * (size_t)i] = o[0]; tmp[3 * (size_t)i + 1] = o[1]; tmp[3 * (size_t)i + 2] = o[2];
}

__global__ void recon_emit_kernel(const double* __restrict__ tmp, const int* __restrict__ flag,
                                  const int* __restrict__ off, int n_max, double* __restrict__ xyz) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_max || !flag[i]) return;
    size_t o = (size_t)off[i];
    xyz[3 * o] = tmp[3 * (size_t)i]; xyz[3 * o + 1] = tmp[3 * (size_t)i + 1]; xyz[3 * o + 2] = tmp[3 * (size_t)i + 2];
}

// ImprovedLaserReconstructor.create_laser_depth_map (improved_reconstruction.py:154-186): depth only at the rounded laser
// pixels.  px = int(round(x)) (half to even), bounds, disparity > 1.0 and not NaN, depth = (fx * baseline) / disparity in
// f64 (np.float64 scalars times an np.float32 element), kept if 0 < depth < 10, stored as f32.  Two points that round to
// the same pixel write the same value (it depends on the pixel's disparity only), so the scatter needs no order.
__global__ void laser_depth_map_kernel(const double* __restrict__ xy, int n, const float* __restrict__ disp, int W, int H,
                                       double fxb, float* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double x = xy[2 * i], y = xy[2 * i + 1];
    if (!(fabs(x) < 2147483647.0 && fabs(y) < 2147483647.0)) return;
    const int px = (int)rint(x), py = (int)rint(y);
    if (px < 0 || px >= W || py < 0 || py >= H) return;
    const float d = disp[(size_t)py * W + px];
    if (!(d > 1.0f) || isnan(d)) return;
    const double depth = __ddiv_rn(fxb, (double)d);
    if (depth > 0 && depth < 10.0) out[(size_t)py * W + px] = (float)depth;
}

int dev_laser_depth_map(Lane& L, const double* xy, int n, const float* disp, int W, int H, double fx, double baseline,
                        float* out) {
    L3D_CHECK(L, cudaMemsetAsync(out, 0, sizeof(float) * (size_t)W * H, L.stream));
    if (n > 0) L3D_LAUNCH(L, laser_depth_map_kernel, cdiv(n, 128), 128, 0, xy, n, disp, W, H, fx * baseline, out);
    return L3D_OK;
}

static bool inv3(const double* m, double* o) {
    double a = m[0], b = m[1], c = m[2], d = m[3], e = m[4], f = m[5], g = m[6], h = m[7], i = m[8];
    double det = a * (e * i - f * h) - b * (d * i - f * g) + c * (d * h - e * g);
    if (det == 0) return false;
    double s = 1.0 / det;
    o[0] = (e * i - f * h) * s; o[1] = (c * h - b * i) * s; o[2] = (b * f - c * e) * s;
    o[3] = (f * g - d * i) * s; o[4] = (a * i - c * g) * s; o[5] = (c * d - a * f) * s;
    o[6] = (d * h - e * g) * s; o[7] = (b * g - a * h) * s; o[8] = (a * e - b * d) * s;
    return true;
}

template <typename T>
int dev_recon(Lane& L, const l3d_recon_params& p, const double* xy, const float* xy_f32, const int* n_dev,
              int n_max, const T* img, int W, int H, double* xyz, int* n_out_dev) {
    L3D_ARG(L, p.kind >= 0 && p.kind <= 3, "recon kind");
    if (std::is_same<T, int16_t>::value) {
        L3D_ARG(L, p.kind == L3D_RECON_DISPARITY || p.kind == L3D_RECON_DISPARITY_MEDIAN, "an int16 disparity map serves the DISPARITY kinds only");
    }
    if (n_max <= 0) { L3D_CHECK(L, cudaMemsetAsync(n_out_dev, 0, sizeof(int), L.stream)); return L3D_OK; }
    ReconArgs a;
    a.p = p;
    memset(a.Kinv, 0, sizeof(a.Kinv));
    if (p.kind == L3D_RECON_PLANE) L3D_ARG(L, inv3(p.K, a.Kinv), "camera matrix is singular");
    if (p.kind == L3D_RECON_DISPARITY_MEDIAN) L3D_ARG(L, recon_window_ok(p.window), "median window must be odd, <= 9");
    if (p.kind != L3D_RECON_PLANE) L3D_ARG(L, img != nullptr, "recon needs a depth/disparity map");
    double* tmp = L.get<double>(S_RC_XYZ, (size_t)n_max * 3);
    int* flag = L.get<int>(S_RC_N, (size_t)n_max * 2);
    int* off = flag + n_max;
    L3D_LAUNCH(L, recon_points_kernel<T>, cdiv(n_max, 128), 128, 0, a, xy, xy_f32, n_dev, n_max, img, W, H, tmp, flag);
    L3D_LAUNCH(L, row_scan_kernel, 1, 1024, 0, flag, n_max, off, n_out_dev);
    L3D_LAUNCH(L, recon_emit_kernel, cdiv(n_max, 128), 128, 0, tmp, flag, off, n_max, xyz);
    return L3D_OK;
}
template int dev_recon<float>(Lane&, const l3d_recon_params&, const double*, const float*, const int*, int, const float*, int,
                              int, double*, int*);
template int dev_recon<int16_t>(Lane&, const l3d_recon_params&, const double*, const float*, const int*, int, const int16_t*,
                                int, int, double*, int*);

}  // namespace l3d
