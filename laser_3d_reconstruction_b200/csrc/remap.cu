// remap.cu -- K1/K1b: fixed-point rectification remap fused with BGR->gray.
// Replaces cv2.remap(img, mapx, mapy, INTER_LINEAR) x2 + cv2.cvtColor(BGR2GRAY) x2
// (camera/single_usb_stereo_camera.py:313-314, 320-321).  Bit-exact: 5 fractional bits,
// weights (32-ay)(32-ax) etc. (sum 1024 == OpenCV's 32768 table / 32), round at half, taps outside
// the source contribute the constant border 0.
// HBM-bound gather: per output pixel 8 B map + <=12 B source taps (L1/L2-resident neighbourhood)
// + 3 B BGR + 1 B gray.  Each thread produces 4 consecutive pixels so the stores are 12 B + 4 B.
#include "common.cuh"

namespace l3d {

// cvRound(v * 32): round-half-even; a non-finite product becomes INT_MIN as x86's cvtss2si makes it, so a NaN or
// infinite map entry saturates to tap -32768 and samples the constant border (cvt.rni would turn NaN into 0, pixel 0)
__device__ __forceinline__ int map_fixed(float v) {
    const float s = __fmul_rn(v, 32.0f);
    return isfinite(s) ? __float2int_rn(s) : INT_MIN;
}

// CV_32FC1 maps -> {ix | iy<<16 (int16 each), ax | ay<<8}
__global__ void build_rectmap_kernel(const float* __restrict__ mx, const float* __restrict__ my, int n, int2* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int sx = map_fixed(mx[i]);
    int sy = map_fixed(my[i]);
    int ix = min(max(sx >> 5, -32768), 32767), iy = min(max(sy >> 5, -32768), 32767);
    int2 o;
    o.x = (ix & 0xffff) | (iy << 16);
    o.y = (sx & 31) | ((sy & 31) << 8);
    out[i] = o;
}

int dev_build_rectmap(Lane& L, const float* mapx_dev, const float* mapy_dev, int W, int H, int2* out) {
    int n = W * H;
    L3D_LAUNCH(L, build_rectmap_kernel, cdiv(n, 256), 256, 0, mapx_dev, mapy_dev, n, out);
    return L3D_OK;
}

__device__ __forceinline__ int gray_of(int b, int g, int r) { return (3735 * b + 19235 * g + 9798 * r + 16384) >> 15; }

__device__ __forceinline__ void remap_px(const uint8_t* __restrict__ src, int sw, int sh, long stride, int2 m, int& b, int& g, int& r) {
    int ix = (int)(short)(m.x & 0xffff), iy = m.x >> 16;
    int ax = m.y & 31, ay = (m.y >> 8) & 31;
    int w00 = (32 - ay) * (32 - ax), w01 = (32 - ay) * ax, w10 = ay * (32 - ax), w11 = ay * ax;
    int sb = 512, sg = 512, sr = 512;
    bool x0 = ix >= 0 && ix < sw, x1 = ix + 1 >= 0 && ix + 1 < sw;
    if (iy >= 0 && iy < sh) {
        const uint8_t* p = src + (long)iy * stride + (long)ix * 3;
        if (x0) { sb += w00 * p[0]; sg += w00 * p[1]; sr += w00 * p[2]; }
        if (x1) { sb += w01 * p[3]; sg += w01 * p[4]; sr += w01 * p[5]; }
    }
    if (iy + 1 >= 0 && iy + 1 < sh) {
        const uint8_t* p = src + (long)(iy + 1) * stride + (long)ix * 3;
        if (x0) { sb += w10 * p[0]; sg += w10 * p[1]; sr += w10 * p[2]; }
        if (x1) { sb += w11 * p[3]; sg += w11 * p[4]; sr += w11 * p[5]; }
    }
    b = sb >> 10; g = sg >> 10; r = sr >> 10;
}

// 4 output pixels per thread (W need not be a multiple of 4; the tail falls back to byte stores)
__global__ void remap_gray_kernel(const uint8_t* __restrict__ src, int sw, int sh, long stride,
                                  const int2* __restrict__ map, int W, int H,
                                  uint8_t* __restrict__ rect, uint8_t* __restrict__ gray) {
    int x4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    int y = blockIdx.y;
    if (x4 >= W) return;
    size_t base = (size_t)y * W + x4;
    int nb = min(4, W - x4);
    uint8_t o[12], gy[4];
    for (int k = 0; k < 4; k++) {
        int b = 0, g = 0, r = 0;
        if (k < nb) remap_px(src, sw, sh, stride, map[base + k], b, g, r);
        o[3 * k] = (uint8_t)b; o[3 * k + 1] = (uint8_t)g; o[3 * k + 2] = (uint8_t)r;
        gy[k] = (uint8_t)gray_of(b, g, r);
    }
    bool vec = (nb == 4) && ((W & 3) == 0);
    if (rect) {
        uint8_t* dst = rect + base * 3;
        if (vec) {
            uint32_t* d32 = (uint32_t*)dst;
            d32[0] = o[0] | (o[1] << 8) | (o[2] << 16) | ((uint32_t)o[3] << 24);
            d32[1] = o[4] | (o[5] << 8) | (o[6] << 16) | ((uint32_t)o[7] << 24);
            d32[2] = o[8] | (o[9] << 8) | (o[10] << 16) | ((uint32_t)o[11] << 24);
        } else for (int k = 0; k < 3 * nb; k++) dst[k] = o[k];
    }
    if (gray) {
        if (vec) *(uint32_t*)(gray + base) = gy[0] | (gy[1] << 8) | (gy[2] << 16) | ((uint32_t)gy[3] << 24);
        else for (int k = 0; k < nb; k++) gray[base + k] = gy[k];
    }
}

int dev_remap_gray(Lane& L, const RectMap& m, const uint8_t* src, int sw, int sh, long stride,
                   uint8_t* rect, uint8_t* gray) {
    L3D_ARG(L, m.map != nullptr, "rectification maps not set");
    L3D_LAUNCH(L, remap_gray_kernel, dim3(cdiv(cdiv(m.W, 4), 64), m.H), 64, 0, src, sw, sh, stride, m.map, m.W, m.H, rect, gray);
    return L3D_OK;
}

// no-rectification branch (map_left_x is None, camera/...:315-317): tight copy + gray
__global__ void copy_gray_kernel(const uint8_t* __restrict__ src, int W, int H, long stride,
                                 uint8_t* __restrict__ bgr, uint8_t* __restrict__ gray) {
    int x = blockIdx.x * blockDim.x + threadIdx.x;
    int y = blockIdx.y;
    if (x >= W) return;
    const uint8_t* p = src + (long)y * stride + (long)x * 3;
    int b = p[0], g = p[1], r = p[2];
    size_t i = (size_t)y * W + x;
    if (bgr) { bgr[3 * i] = (uint8_t)b; bgr[3 * i + 1] = (uint8_t)g; bgr[3 * i + 2] = (uint8_t)r; }
    if (gray) gray[i] = (uint8_t)gray_of(b, g, r);
}

int dev_copy_gray(Lane& L, const uint8_t* src, int W, int H, long stride, uint8_t* bgr, uint8_t* gray) {
    L3D_LAUNCH(L, copy_gray_kernel, dim3(cdiv(W, 128), H), 128, 0, src, W, H, stride, bgr, gray);
    return L3D_OK;
}

// ---- cv2.initUndistortRectifyMap(K, dist, R, P, size, CV_32FC1) (camera/single_usb_stereo_camera.py:190-206; SURVEY 8f N3)
// per destination pixel, f64, every operation rounded on its own in cv2's order (restated and pinned against cv2 in
// oracle/ref_ops.py::init_undistort_rectify_map): [x y w] = iR [u v 1], x/w, y/w, rational radial + tangential +
// thin-prism distortion, projection with K, stored as f32.  iR = (P[:3,:3] R)^-1 comes from the caller.
struct UndistArgs { double ir[9]; double k[12]; double fx, fy, u0, v0; };

__global__ void init_undistort_map_kernel(UndistArgs a, int W, int H, float* __restrict__ mapx, float* __restrict__ mapy) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (j >= W) return;
    const double di = (double)i, dj = (double)j;
    const double _x = __dadd_rn(__dadd_rn(__dmul_rn(di, a.ir[1]), a.ir[2]), __dmul_rn(dj, a.ir[0]));
    const double _y = __dadd_rn(__dadd_rn(__dmul_rn(di, a.ir[4]), a.ir[5]), __dmul_rn(dj, a.ir[3]));
    const double _w = __dadd_rn(__dadd_rn(__dmul_rn(di, a.ir[7]), a.ir[8]), __dmul_rn(dj, a.ir[6]));
    const double w = __ddiv_rn(1.0, _w);
    const double x = __dmul_rn(_x, w), y = __dmul_rn(_y, w);
    const double x2 = __dmul_rn(x, x), y2 = __dmul_rn(y, y);
    const double r2 = __dadd_rn(x2, y2), _2xy = __dmul_rn(__dmul_rn(2.0, x), y);
    const double k1 = a.k[0], k2 = a.k[1], p1 = a.k[2], p2 = a.k[3], k3 = a.k[4], k4 = a.k[5], k5 = a.k[6], k6 = a.k[7];
    const double s1 = a.k[8], s2 = a.k[9], s3 = a.k[10], s4 = a.k[11];
    const double num = __dadd_rn(1.0, __dmul_rn(__dadd_rn(__dmul_rn(__dadd_rn(__dmul_rn(k3, r2), k2), r2), k1), r2));
    const double den = __dadd_rn(1.0, __dmul_rn(__dadd_rn(__dmul_rn(__dadd_rn(__dmul_rn(k6, r2), k5), r2), k4), r2));
    const double kr = __ddiv_rn(num, den);
    double xd = __dadd_rn(__dmul_rn(x, kr), __dmul_rn(p1, _2xy));
    xd = __dadd_rn(xd, __dmul_rn(p2, __dadd_rn(r2, __dmul_rn(2.0, x2))));
    xd = __dadd_rn(xd, __dmul_rn(s1, r2));
    xd = __dadd_rn(xd, __dmul_rn(__dmul_rn(s2, r2), r2));
    double yd = __dadd_rn(__dmul_rn(y, kr), __dmul_rn(p1, __dadd_rn(r2, __dmul_rn(2.0, y2))));
    yd = __dadd_rn(yd, __dmul_rn(p2, _2xy));
    yd = __dadd_rn(yd, __dmul_rn(s3, r2));
    yd = __dadd_rn(yd, __dmul_rn(__dmul_rn(s4, r2), r2));
    const size_t o = (size_t)i * W + j;
    mapx[o] = (float)__dadd_rn(__dmul_rn(a.fx, xd), a.u0);
    mapy[o] = (float)__dadd_rn(__dmul_rn(a.fy, yd), a.v0);
}

int dev_init_undistort_map(Lane& L, const double* K, const double* dist, int ndist, const double* iR, int W, int H,
                           float* mapx, float* mapy) {
    L3D_ARG(L, ndist >= 0 && ndist <= 14, "initUndistortRectifyMap: at most 14 distortion coefficients");
    UndistArgs a;
    for (int i = 0; i < 9; i++) a.ir[i] = iR[i];
    for (int i = 0; i < 12; i++) a.k[i] = i < ndist ? dist[i] : 0.0;
    if (ndist > 12 && (dist[12] != 0.0 || (ndist > 13 && dist[13] != 0.0))) {
        set_err(L.err, "initUndistortRectifyMap: tilted-sensor coefficients are not supported");
        return L3D_ERR_UNSUPPORTED;
    }
    a.fx = K[0]; a.fy = K[4]; a.u0 = K[2]; a.v0 = K[5];
    L3D_LAUNCH(L, init_undistort_map_kernel, dim3(cdiv(W, 128), H), 128, 0, a, W, H, mapx, mapy);
    return L3D_OK;
}

}  // namespace l3d
