// api.cu -- the C ABI of include/l3d.h: context, host<->device marshalling, single-frame calls (the frame pipeline's
// entry points are in pipeline.cu).
#include <stdexcept>

#include <nvtx3/nvToolsExt.h>

#include "api.cuh"

namespace l3d {

static std::string g_create_err;

void set_err(std::string* err, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (err) *err = buf;
}

void* Lane::get(Slot s, size_t bytes) {
    DevBuf& b = bufs[s];
    if (bytes == 0) bytes = 16;
    if (b.cap >= bytes) return b.p;
    if (b.p) {
        cudaStreamSynchronize(stream);  // earlier work may still read the old buffer
        cudaFree(b.p);
        b.p = nullptr; b.cap = 0;
    }
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) {
        b.p = nullptr;
        char msg[256];
        snprintf(msg, sizeof(msg), "cudaMalloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
        throw std::runtime_error(msg);
    }
    b.cap = want;
    return b.p;
}

void Lane::release() {
    if (stream) cudaStreamSynchronize(stream);
    for (auto& b : bufs) { if (b.p) cudaFree(b.p); b.p = nullptr; b.cap = 0; }
    for (auto e : ev_pool) cudaEventDestroy(e);
    ev_pool.clear(); timers.clear(); ev_used = 0;
    if (stream) { cudaStreamDestroy(stream); stream = nullptr; }
    if (back_stream) { cudaStreamSynchronize(back_stream); cudaStreamDestroy(back_stream); back_stream = nullptr; }
    if (back_done) { cudaEventDestroy(back_done); back_done = nullptr; }
}

cudaEvent_t Lane::new_event() {
    if (ev_used == ev_pool.size()) { cudaEvent_t e; cudaEventCreate(&e); ev_pool.push_back(e); }
    return ev_pool[ev_used++];
}
// Kernel groups (sgbm_cost, sgbm_scan_k*, sgbm_vgroup_*, sgbm_wta, wls, remap, extract, recon) are bracketed by NVTX ranges
// when L3D_NVTX=1 (host-side push/pop around the enqueue: they show up as ranges over the launches in Nsight Systems /
// ncu --nvtx) and by CUDA events when timing is on (bench roofline leg).
static bool nvtx_on() {
    static const bool on = getenv("L3D_NVTX") && atoi(getenv("L3D_NVTX")) > 0;
    return on;
}
void Lane::t_begin(const char* name) {
    if (nvtx_on()) nvtxRangePushA(name);
    if (!timing) return;
    TimerRec r; r.a = new_event(); r.b = nullptr;
    cudaEventRecord(r.a, stream);
    timers[name].push_back(r);
}
void Lane::t_end(const char* name) {
    if (nvtx_on()) nvtxRangePop();
    if (!timing) return;
    auto& v = timers[name];
    if (v.empty() || v.back().b) return;
    v.back().b = new_event();
    cudaEventRecord(v.back().b, stream);
}
void Lane::t_reset() { timers.clear(); ev_used = 0; }

int check_flags(l3d_ctx* ctx, unsigned* flags) {
    if (!flags) return L3D_OK;
    unsigned h = 0;
    if (cudaMemcpy(&h, flags, sizeof(unsigned), cudaMemcpyDeviceToHost) != cudaSuccess) { cudaGetLastError(); return L3D_OK; }
    if (!h) return L3D_OK;
    cudaMemset(flags, 0, sizeof(unsigned));
    set_err(&ctx->err, "StereoSGBM: the cost volume left the int16 value domain (block sum + P2 >= 32768); cv2 wraps there, "
                       "this input is not supported");
    return L3D_ERR_UNSUPPORTED;
}

int set_maps(l3d_ctx* ctx, Lane& L, RectMap& m, const float* mapx, const float* mapy, int W, int H) {
    size_t n = (size_t)W * H;
    float* tmp = L.get<float>(S_IO_A, 2 * n);
    CK(ctx, cudaMemcpyAsync(tmp, mapx, n * 4, cudaMemcpyHostToDevice, L.stream));
    CK(ctx, cudaMemcpyAsync(tmp + n, mapy, n * 4, cudaMemcpyHostToDevice, L.stream));
    if (m.map) { CK(ctx, cudaStreamSynchronize(L.stream)); cudaFree(m.map); m.map = nullptr; }
    CK(ctx, cudaMalloc(&m.map, n * sizeof(int2)));
    m.W = W; m.H = H;
    RC(dev_build_rectmap(L, tmp, tmp + n, W, H, m.map));
    CK(ctx, cudaStreamSynchronize(L.stream));
    return L3D_OK;
}

int depth_front(Lane& L, const l3d_depth_config& cfg, const RectMap* maps, const uint8_t* lsrc, const uint8_t* rsrc,
                int W, int H, long stride, uint8_t* rectL, DepthRuns& dr) {
    size_t n = (size_t)W * H;
    uint8_t* gl = L.get<uint8_t>(S_GRAY_L, n);
    uint8_t* gr = L.get<uint8_t>(S_GRAY_R, n);
    L.t_begin("remap");
    if (cfg.use_maps) {
        L3D_ARG(L, maps[0].map && maps[1].map, "rectification maps not set");
        L3D_ARG(L, maps[0].W == W && maps[0].H == H && maps[1].W == W && maps[1].H == H, "map size != image size");
        RC(dev_remap_gray(L, maps[0], lsrc, W, H, stride, rectL, gl));
        RC(dev_remap_gray(L, maps[1], rsrc, W, H, stride, nullptr, gr));
    } else {
        RC(dev_copy_gray(L, lsrc, W, H, stride, rectL, gl));
        RC(dev_copy_gray(L, rsrc, W, H, stride, nullptr, gr));
    }
    L.t_end("remap");
    uint4* dL = L.get<uint4>(S_DESC_L, 2 * n);  // two operand planes per view (sgbm_prefilter_kernel)
    uint4* dR = L.get<uint4>(S_DESC_R, 2 * n);
    dr.has_right = cfg.use_wls != 0;
    dr.left.no_hpair = dr.right.no_hpair = dr.vwave;
    // the right matcher sees the views swapped: same BT operands, roles exchanged, one pixel-cost pass for both volumes
    if (dr.has_right) RC(sgbm_front_pair(L, cfg.left, cfg.right, gl, gr, W, H, dL, dR, dr.left, dr.right));
    else RC(sgbm_front(L, cfg.left, gl, gr, W, H, 0, dL, dR, true, dr.left));
    return L3D_OK;
}

int depth_back(Lane& L, const l3d_depth_config& cfg, DepthRuns& dr, int W, int H, float* depth, int16_t* disp_f) {
    size_t n = (size_t)W * H;
    const uint8_t* gl = L.get<uint8_t>(S_GRAY_L, n);
    int16_t* dl = L.get<int16_t>(S_DISP_L, n);
    RC(sgbm_back(L, dr.left, dl, nullptr));
    const double* Q = cfg.use_Q ? cfg.Q : nullptr;
    if (dr.has_right) {
        int16_t* drr = L.get<int16_t>(S_DISP_R, n);
        RC(sgbm_back(L, dr.right, drr, nullptr));
        return dev_wls(L, cfg.wls, dl, drr, gl, W, H, disp_f, nullptr, depth, Q);  // the filter's last kernel writes the depth too
    }
    L3D_CHECK(L, cudaMemcpyAsync(disp_f, dl, n * 2, cudaMemcpyDeviceToDevice, L.stream));
    return dev_depth(L, dl, W, H, Q, depth);
}

// the previous-row paths run direction-split: a lone volume would occupy 8 SMs in the cluster kernel
int depth_rest(Lane& L, const l3d_depth_config& cfg, DepthRuns& dr, int W, int H, float* depth, int16_t* disp_f) {
    RC(sgbm_middle_split(L, dr.left, false));
    if (dr.has_right) RC(sgbm_middle_split(L, dr.right, false));
    return depth_back(L, cfg, dr, W, H, depth, disp_f);
}

}  // namespace l3d

using namespace l3d;

extern "C" {

const char* l3d_version(void) { return "laser3d-b200 0.1 (sm_100a)"; }

// The frame pipeline keeps 14+ streams busy; with the default of 8 hardware work queues streams share queues
// and serialise falsely.  Must be in the environment before the process creates its CUDA context (a host
// application that initialises CUDA first has to export it itself); never overrides the user's value.
static void want_hw_queues() { setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0); }

int l3d_device_count(void) {
    want_hw_queues();
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int l3d_ctx_create(int device, l3d_ctx** out) {
    if (!out) return L3D_ERR_ARG;
    *out = nullptr;
    want_hw_queues();
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        set_err(&g_create_err, "no CUDA device available (%s); this library has no CPU fallback",
                e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        cudaGetLastError();
        return L3D_ERR_CUDA;
    }
    if (device < 0 || device >= n) { set_err(&g_create_err, "device %d out of range [0,%d)", device, n); return L3D_ERR_ARG; }
    e = cudaSetDevice(device);
    if (e != cudaSuccess) { set_err(&g_create_err, "cudaSetDevice(%d): %s", device, cudaGetErrorString(e)); return L3D_ERR_CUDA; }
    l3d_ctx* c = new l3d_ctx();
    c->device = device;
    c->stager = new HostStager();
    c->lane.err = &c->err;
    e = cudaStreamCreateWithFlags(&c->lane.stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { set_err(&g_create_err, "cudaStreamCreate: %s", cudaGetErrorString(e)); delete c->stager; delete c; return L3D_ERR_CUDA; }
    e = cudaMalloc(&c->lane.flags, 16);
    if (e == cudaSuccess) e = cudaMemset(c->lane.flags, 0, 16);
    if (e != cudaSuccess) { set_err(&g_create_err, "cudaMalloc: %s", cudaGetErrorString(e)); delete c->stager; delete c; return L3D_ERR_CUDA; }
    *out = c;
    return L3D_OK;
}

void l3d_ctx_destroy(l3d_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    ctx->lane.release();
    if (ctx->lane.flags) cudaFree(ctx->lane.flags);
    for (auto& m : ctx->maps) if (m.map) cudaFree(m.map);
    delete ctx->stager;
    delete ctx;
}

const char* l3d_last_error(l3d_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

int l3d_sync(l3d_ctx* ctx) {
    if (!ctx) return L3D_ERR_ARG;
    CK(ctx, cudaStreamSynchronize(ctx->lane.stream));
    return L3D_OK;
}

long long l3d_launch_count(l3d_ctx* ctx) { return ctx ? ctx->lane.launches : 0; }

// ---- small helpers -----------------------------------------------------------------------
// Host <-> device copies of the single-frame calls.  Large ones are staged through the context's page-locked arena with a
// few copy threads (hostcopy.cuh); a staged d2h lands in the caller's memory in finish(), which every call ends with.
static int h2d(l3d_ctx* ctx, void* dst, const void* src, size_t bytes) {
    if (ctx->stager->wants(bytes)) CK(ctx, ctx->stager->h2d(dst, src, bytes, ctx->lane.stream));
    else CK(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->lane.stream));
    return L3D_OK;
}
static int d2h(l3d_ctx* ctx, void* dst, const void* src, size_t bytes) {
    if (ctx->stager->wants(bytes)) CK(ctx, ctx->stager->d2h(dst, src, bytes, ctx->lane.stream));
    else CK(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->lane.stream));
    return L3D_OK;
}
static int finish(l3d_ctx* ctx) {
    CK(ctx, ctx->stager->finish(ctx->lane.stream));
    return L3D_OK;
}

int l3d_set_rectify_maps(l3d_ctx* ctx, int eye, const float* mapx, const float* mapy, int W, int H) {
    API_BEGIN(ctx)
    NEED(ctx, eye == 0 || eye == 1, "eye must be 0 (left) or 1 (right)");
    NEED(ctx, mapx && mapy && W > 0 && H > 0, "maps");
    CK(ctx, cudaSetDevice(ctx->device));
    return set_maps(ctx, ctx->lane, ctx->maps[eye], mapx, mapy, W, H);
    API_END(ctx)
}

int l3d_remap_gray(l3d_ctx* ctx, int eye, const uint8_t* src_bgr, int sw, int sh, long src_stride,
                   uint8_t* rect_bgr, uint8_t* gray) {
    API_BEGIN(ctx)
    NEED(ctx, eye == 0 || eye == 1, "eye");
    NEED(ctx, src_bgr && sw > 0 && sh > 0 && src_stride >= 3L * sw, "source image");
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = ctx->lane;
    const RectMap& m = ctx->maps[eye];
    NEED(ctx, m.map, "rectification maps not set for this eye");
    // a strided view (the halves _split_frame returns) ends with its last ROW, not with a whole stride
    size_t nsrc = (size_t)src_stride * (sh - 1) + 3 * (size_t)sw, n = (size_t)m.W * m.H;
    uint8_t* s = L.get<uint8_t>(S_SRC_L, nsrc);
    uint8_t* r = L.get<uint8_t>(S_RECT_L, n * 3);
    uint8_t* g = L.get<uint8_t>(S_GRAY_L, n);
    RC(h2d(ctx, s, src_bgr, nsrc));
    RC(dev_remap_gray(L, m, s, sw, sh, src_stride, r, g));
    if (rect_bgr) RC(d2h(ctx, rect_bgr, r, n * 3));
    if (gray) RC(d2h(ctx, gray, g, n));
    RC(finish(ctx));
    return L3D_OK;
    API_END(ctx)
}

int l3d_bgr2gray(l3d_ctx* ctx, const uint8_t* bgr, int W, int H, uint8_t* gray) {
    API_BEGIN(ctx)
    NEED(ctx, bgr && gray && W > 0 && H > 0, "image");
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = ctx->lane;
    size_t n = (size_t)W * H;
    uint8_t* s = L.get<uint8_t>(S_SRC_L, n * 3);
    uint8_t* g = L.get<uint8_t>(S_GRAY_L, n);
    RC(h2d(ctx, s, bgr, n * 3));
    RC(dev_copy_gray(L, s, W, H, 3L * W, nullptr, g));
    RC(d2h(ctx, gray, g, n));
    RC(finish(ctx));
    return L3D_OK;
    API_END(ctx)
}

int l3d_sgbm_volume_rows(const l3d_sgbm_params* p, int W, int H) { return p ? sgbm_volume_rows(*p, W, H) : -1; }

int l3d_sgbm_debug(l3d_ctx* ctx, const l3d_sgbm_params* p, const uint8_t* left, const uint8_t* right,
                   int W, int H, int16_t* disp, int16_t* raw, int16_t* C_out, int16_t* S_out) {
    API_BEGIN(ctx)
    NEED(ctx, p && left && right && disp && W > 0 && H > 0, "sgbm arguments");
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = ctx->lane;
    size_t n = (size_t)W * H;
    uint8_t* l = L.get<uint8_t>(S_GRAY_L, n);
    uint8_t* r = L.get<uint8_t>(S_GRAY_R, n);
    int16_t* d = L.get<int16_t>(S_DISP_L, n);
    RC(h2d(ctx, l, left, n));
    RC(h2d(ctx, r, right, n));
    SgbmDebug dbg;
    size_t nvol = 0;
    if (C_out || S_out) {
        int hv = sgbm_volume_rows(*p, W, H);
        NEED(ctx, hv > 0, "sgbm parameters");
        const int width1 = sgbm_width1(*p, W);
        nvol = width1 > 0 ? (size_t)hv * width1 * p->numDisparities : 0;
        if (nvol) {
            int16_t* vols = L.get<int16_t>(S_IO_B, nvol * 2);
            if (C_out) dbg.C = vols;
            if (S_out) dbg.S = vols + nvol;
        }
    }
    if (raw) dbg.raw = L.get<int16_t>(S_IO_C, n);
    RC(dev_sgbm(L, *p, l, r, W, H, d, &dbg));
    RC(d2h(ctx, disp, d, n * 2));
    if (raw) RC(d2h(ctx, raw, dbg.raw, n * 2));
    if (C_out && dbg.C) RC(d2h(ctx, C_out, dbg.C, nvol * 2));
    if (S_out && dbg.S) RC(d2h(ctx, S_out, dbg.S, nvol * 2));
    RC(finish(ctx));
    return check_flags(ctx, L.flags);
    API_END(ctx)
}

int l3d_sgbm_compute_pair(l3d_ctx* ctx, const l3d_sgbm_params* pl, const l3d_sgbm_params* pr, const uint8_t* left,
                          const uint8_t* right, int W, int H, int16_t* disp_left, int16_t* disp_right, int16_t* Cl_out,
                          int16_t* Cr_out) {
    API_BEGIN(ctx)
    NEED(ctx, pl && pr && left && right && disp_left && disp_right && W > 0 && H > 0, "sgbm pair arguments");
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = ctx->lane;
    size_t n = (size_t)W * H;
    uint8_t* l = L.get<uint8_t>(S_GRAY_L, n);
    uint8_t* r = L.get<uint8_t>(S_GRAY_R, n);
    int16_t* dl = L.get<int16_t>(S_DISP_L, n);
    int16_t* dr = L.get<int16_t>(S_DISP_R, n);
    uint4* dL = L.get<uint4>(S_DESC_L, 2 * n);
    uint4* dR = L.get<uint4>(S_DESC_R, 2 * n);
    RC(h2d(ctx, l, left, n));
    RC(h2d(ctx, r, right, n));
    SgbmRun rl, rr;
    RC(sgbm_front_pair(L, *pl, *pr, l, r, W, H, dL, dR, rl, rr));
    if (Cl_out && rl.C) RC(d2h(ctx, Cl_out, rl.C, (size_t)rl.g.HV * rl.g.width1 * rl.g.D * 2));
    if (Cr_out && rr.C) RC(d2h(ctx, Cr_out, rr.C, (size_t)rr.g.HV * rr.g.width1 * rr.g.D * 2));
    RC(sgbm_middle_split(L, rl, false));
    RC(sgbm_middle_split(L, rr, false));
    RC(sgbm_back(L, rl, dl, nullptr));
    RC(sgbm_back(L, rr, dr, nullptr));
    RC(d2h(ctx, disp_left, dl, n * 2));
    RC(d2h(ctx, disp_right, dr, n * 2));
    RC(finish(ctx));
    return check_flags(ctx, L.flags);
    API_END(ctx)
}

int l3d_sgbm_compute(l3d_ctx* ctx, const l3d_sgbm_params* p, const uint8_t* left, const uint8_t* right,
                     int W, int H, int16_t* disp) {
    return l3d_sgbm_debug(ctx, p, left, right, W, H, disp, nullptr, nullptr, nullptr);
}

static int cloud_op(l3d_ctx* ctx, const double* points, int n, double* out, int* n_out, int op, double a, int k, int f32) {
    API_BEGIN(ctx)
    NEED(ctx, n >= 0 && n_out && (n == 0 || (points && out)), "point cloud arguments");
    *n_out = 0;
    if (n == 0) return L3D_OK;
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = ctx->lane;
    double* dp = L.get<double>(S_RC_XY, (size_t)n * 3);
    double* dout = L.get<double>(S_RC_XYZ, (size_t)n * 3);
    RC(h2d(ctx, dp, points, (size_t)n * 24));
    int m = 0;
    if (op == 0) RC(dev_voxel_downsample(L, dp, n, a, f32, dout, &m));
    else RC(dev_outlier_removal(L, dp, n, k, a, dout, &m));
    if (m > 0) RC(d2h(ctx, out, dout, (size_t)m * 24));
    RC(finish(ctx));
    *n_out = m;
    return L3D_OK;
    API_END(ctx)
}
int l3d_voxel_downsample(l3d_ctx* ctx, const double* points, int n, double voxel_size, int f32_arithmetic, double* out,
                         int* n_out) {
    return cloud_op(ctx, points, n, out, n_out, 0, voxel_size, 0, f32_arithmetic);
}
int l3d_statistical_outlier_removal(l3d_ctx* ctx, const double* points, int n, int nb_neighbors, double std_ratio,
                                    double* out, int* n_out) {
    return cloud_op(ctx, points, n, out, n_out, 1, std_ratio, nb_neighbors, 0);
}

int l3d_init_undistort_rectify_map(l3d_ctx* ctx, const double* K, const double* dist, int ndist, const double* iR,
                                   int W, int H, float* mapx, float* mapy) {
    API_BEGIN(ctx)
    NEED(ctx, K && iR && mapx && mapy && W > 0 && H > 0 && (dist || ndist == 0), "initUndistortRectifyMap arguments");
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = ctx->lane;
    size_t n = (size_t)W * H;
    float* mx = L.get<float>(S_IO_A, n);
    float* my = L.get<float>(S_IO_B, n);
    RC(dev_init_undistort_map(L, K, dist, ndist, iR, W, H, mx, my));
    RC(d2h(ctx, mapx, mx, n * 4));
    RC(d2h(ctx, mapy, my, n * 4));
    RC(finish(ctx));
    return L3D_OK;
    API_END(ctx)
}

int l3d_bm_compute(l3d_ctx* ctx, const l3d_bm_params* p, const uint8_t* left, const uint8_t* right, int W, int H,
                   int16_t* disp) {
    API_BEGIN(ctx)
    NEED(ctx, p && left && right && disp && W > 0 && H > 0, "StereoBM arguments");
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = ctx->lane;
    size_t n = (size_t)W * H;
    uint8_t* l = L.get<uint8_t>(S_GRAY_L, n);
    uint8_t* r = L.get<uint8_t>(S_GRAY_R, n);
    int16_t* d = L.get<int16_t>(S_DISP_L, n);
    RC(h2d(ctx, l, left, n));
    RC(h2d(ctx, r, right, n));
    RC(dev_bm(L, *p, l, r, W, H, d));
    RC(d2h(ctx, disp, d, n * 2));
    RC(finish(ctx));
    return L3D_OK;
    API_END(ctx)
}

int l3d_median3_s16(l3d_ctx* ctx, const int16_t* src, int W, int H, int16_t* dst) {
    API_BEGIN(ctx)
    NEED(ctx, src && dst && W > 0 && H > 0, "image");
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = ctx->lane;
    size_t n = (size_t)W * H;
    int16_t* a = L.get<int16_t>(S_DISP_L, n);
    int16_t* b = L.get<int16_t>(S_DISP_R, n);
    RC(h2d(ctx, a, src, n * 2));
    RC(dev_median3(L, a, W, H, b));
    RC(d2h(ctx, dst, b, n * 2));
    RC(finish(ctx));
    return L3D_OK;
    API_END(ctx)
}

int l3d_filter_speckles(l3d_ctx* ctx, int16_t* img, int W, int H, int newVal, int maxSize, int maxDiff) {
    API_BEGIN(ctx)
    NEED(ctx, img && W > 0 && H > 0, "image");
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = ctx->lane;
    size_t n = (size_t)W * H;
    int16_t* a = L.get<int16_t>(S_DISP_L, n);
    RC(h2d(ctx, a, img, n * 2));
    RC(dev_speckles(L, a, W, H, newVal, maxSize, maxDiff));
    RC(d2h(ctx, img, a, n * 2));
    RC(finish(ctx));
    return L3D_OK;
    API_END(ctx)
}

int l3d_wls_filter(l3d_ctx* ctx, const l3d_wls_params* p, const int16_t* dl, const int16_t* dr,
                   const uint8_t* guide, int W, int H, int16_t* out, float* conf_out) {
    API_BEGIN(ctx)
    NEED(ctx, p && dl && dr && guide && out && W > 0 && H > 0, "wls arguments");
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = ctx->lane;
    size_t n = (size_t)W * H;
    int16_t* a = L.get<int16_t>(S_DISP_L, n);
    int16_t* b = L.get<int16_t>(S_DISP_R, n);
    int16_t* o = L.get<int16_t>(S_DISP_F, n);
    uint8_t* g = L.get<uint8_t>(S_GRAY_L, n);
    float* cf = conf_out ? L.get<float>(S_IO_A, n) : nullptr;
    RC(h2d(ctx, a, dl, n * 2));
    RC(h2d(ctx, b, dr, n * 2));
    RC(h2d(ctx, g, guide, n));
    RC(dev_wls(L, *p, a, b, g, W, H, o, cf));
    RC(d2h(ctx, out, o, n * 2));
    if (conf_out) RC(d2h(ctx, conf_out, cf, n * 4));
    RC(finish(ctx));
    return L3D_OK;
    API_END(ctx)
}

int l3d_fgs_solve(l3d_ctx* ctx, int solver, int variant, double lambda, int iters, const float* ch, const float* cv,
                  int w, int h, float* num, float* den, int* parallel_used) {
    API_BEGIN(ctx)
    NEED(ctx, ch && cv && num && den && w > 0 && h > 0, "fgs arguments");
    NEED(ctx, iters >= 1 && iters <= 3, "fgs iters (1..3)");
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = ctx->lane;
    size_t n = (size_t)w * h;
    // the planes dev_wls solves in
    float *a = L.get<float>(S_WLS_A, n), *b = L.get<float>(S_WLS_B, n), *D = L.get<float>(S_WLS_C, n);
    float *wh = L.get<float>(S_WLS_H, n), *wv = L.get<float>(S_WLS_I, n);
    RC(h2d(ctx, a, num, n * 4));
    RC(h2d(ctx, b, den, n * 4));
    RC(h2d(ctx, wh, ch, n * 4));
    RC(h2d(ctx, wv, cv, n * 4));
    bool par = false;
    RC(dev_fgs(L, solver, variant, lambda, iters, wh, wv, w, h, a, b, D, &par));
    RC(d2h(ctx, num, a, n * 4));
    RC(d2h(ctx, den, b, n * 4));
    RC(finish(ctx));
    if (parallel_used) *parallel_used = par ? 1 : 0;
    return L3D_OK;
    API_END(ctx)
}

int l3d_disp_to_depth(l3d_ctx* ctx, const int16_t* disp16, int W, int H, const double* Q, float* depth) {
    API_BEGIN(ctx)
    NEED(ctx, disp16 && depth && W > 0 && H > 0, "depth arguments");
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = ctx->lane;
    size_t n = (size_t)W * H;
    int16_t* a = L.get<int16_t>(S_DISP_F, n);
    float* d = L.get<float>(S_DEPTH, n);
    RC(h2d(ctx, a, disp16, n * 2));
    RC(dev_depth(L, a, W, H, Q, d));
    RC(d2h(ctx, depth, d, n * 4));
    RC(finish(ctx));
    return L3D_OK;
    API_END(ctx)
}

int l3d_compute_depth(l3d_ctx* ctx, const l3d_depth_config* cfg, const uint8_t* left_bgr, const uint8_t* right_bgr,
                      int W, int H, long stride, uint8_t* left_rect, float* depth, int16_t* disp_out) {
    API_BEGIN(ctx)
    NEED(ctx, cfg && left_bgr && right_bgr && depth && W > 0 && H > 0 && stride >= 3L * W, "compute_depth arguments");
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = ctx->lane;
    size_t n = (size_t)W * H, ns = (size_t)stride * (H - 1) + 3 * (size_t)W;  // strided views end with their last row
    uint8_t* sl = L.get<uint8_t>(S_SRC_L, ns);
    uint8_t* sr = L.get<uint8_t>(S_SRC_R, ns);
    uint8_t* rl = L.get<uint8_t>(S_RECT_L, n * 3);
    float* dp = L.get<float>(S_DEPTH, n);
    int16_t* df = L.get<int16_t>(S_DISP_F, n);
    RC(h2d(ctx, sl, left_bgr, ns));
    RC(h2d(ctx, sr, right_bgr, ns));
    // the rectified view goes back as soon as it exists: its DMA and the copy into the caller's array run under the matchers
    DepthRuns dr;
    RC(depth_front(L, *cfg, ctx->maps, sl, sr, W, H, stride, rl, dr));
    if (left_rect) RC(d2h(ctx, left_rect, rl, n * 3));
    RC(depth_rest(L, *cfg, dr, W, H, dp, df));
    RC(d2h(ctx, depth, dp, n * 4));
    if (disp_out) RC(d2h(ctx, disp_out, df, n * 2));
    RC(finish(ctx));
    return check_flags(ctx, L.flags);
    API_END(ctx)
}

int l3d_simple_extract(l3d_ctx* ctx, const uint8_t* bgr, int W, int H, const int* hsv_lo, const int* hsv_hi,
                       int bright_thr, double min_area, uint8_t* mask_morph, uint8_t* mask_final, double* xy, int* n) {
    API_BEGIN(ctx)
    NEED(ctx, bgr && hsv_lo && hsv_hi && xy && n && W > 0 && H > 0, "simple_extract arguments");
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = ctx->lane;
    size_t np = (size_t)W * H;
    uint8_t* s = L.get<uint8_t>(S_SRC_L, np * 3);
    uint8_t* mm = L.get<uint8_t>(S_IO_A, np * 2);
    double* dxy = L.get<double>(S_SM_XY, (size_t)2 * H + 2);
    int* dn = (int*)L.get(S_ST_N, 16);
    RC(h2d(ctx, s, bgr, np * 3));
    RC(dev_simple(L, s, W, H, hsv_lo, hsv_hi, bright_thr, min_area, mask_morph ? mm : nullptr,
                  mask_final ? mm + np : nullptr, dxy, dn));
    RC(d2h(ctx, n, dn, sizeof(int)));
    if (mask_morph) RC(d2h(ctx, mask_morph, mm, np));
    if (mask_final) RC(d2h(ctx, mask_final, mm + np, np));
    RC(finish(ctx));
    if (*n > 0) { RC(d2h(ctx, xy, dxy, sizeof(double) * 2 * (size_t)*n)); RC(finish(ctx)); }
    return L3D_OK;
    API_END(ctx)
}

int l3d_steger_extract(l3d_ctx* ctx, const l3d_steger_params* p, const uint8_t* img, int channels, int W, int H,
                       float* xy, int cap, int* n) {
    API_BEGIN(ctx)
    NEED(ctx, p && img && xy && n && cap >= 0 && W > 0 && H > 0, "steger_extract arguments");
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = ctx->lane;
    size_t nb = (size_t)W * H * channels;
    uint8_t* s = L.get<uint8_t>(S_SRC_L, nb);
    float* dxy = L.get<float>(S_ST_XY, (size_t)2 * std::max(cap, 1));
    int* dn = (int*)L.get(S_ST_N, 16);
    RC(h2d(ctx, s, img, nb));
    RC(dev_steger(L, *p, s, channels, W, H, dxy, cap, dn));
    RC(d2h(ctx, n, dn, sizeof(int)));
    RC(finish(ctx));
    int m = std::min(*n, cap);
    if (m > 0) { RC(d2h(ctx, xy, dxy, sizeof(float) * 2 * (size_t)m)); RC(finish(ctx)); }
    return L3D_OK;
    API_END(ctx)
}

int l3d_reconstruct(l3d_ctx* ctx, const l3d_recon_params* p, const double* xy, int n, const float* img, int W,
                    int H, double* xyz, int* n_out) {
    API_BEGIN(ctx)
    NEED(ctx, p && n_out && n >= 0, "reconstruct arguments");
    *n_out = 0;
    if (n == 0) return L3D_OK;
    NEED(ctx, xy && xyz, "reconstruct buffers");
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = ctx->lane;
    double* dxy = L.get<double>(S_RC_XY, (size_t)2 * n);
    double* dxyz = L.get<double>(S_IO_D, (size_t)3 * n);
    int* dn = (int*)L.get(S_IO_E, 16);
    float* dimg = nullptr;
    if (p->kind != L3D_RECON_PLANE) {
        NEED(ctx, img && W > 0 && H > 0, "reconstruct needs a depth/disparity map");
        dimg = L.get<float>(S_DEPTH, (size_t)W * H);
        RC(h2d(ctx, dimg, img, (size_t)W * H * 4));
    }
    RC(h2d(ctx, dxy, xy, sizeof(double) * 2 * (size_t)n));
    RC(dev_recon(L, *p, dxy, nullptr, nullptr, n, dimg, W, H, dxyz, dn));
    RC(d2h(ctx, n_out, dn, sizeof(int)));
    RC(finish(ctx));
    if (*n_out > 0) { RC(d2h(ctx, xyz, dxyz, sizeof(double) * 3 * (size_t)*n_out)); RC(finish(ctx)); }
    return L3D_OK;
    API_END(ctx)
}

int l3d_laser_depth_map(l3d_ctx* ctx, const double* xy, int n, const float* disp, int W, int H, double fx,
                        double baseline, float* out) {
    API_BEGIN(ctx)
    NEED(ctx, n >= 0 && disp && out && W > 0 && H > 0 && (n == 0 || xy), "laser_depth_map arguments");
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = ctx->lane;
    const size_t np = (size_t)W * H;
    float* dimg = L.get<float>(S_DEPTH, np);
    float* dout = L.get<float>(S_IO_D, np);
    double* dxy = L.get<double>(S_RC_XY, (size_t)2 * std::max(n, 1));
    RC(h2d(ctx, dimg, disp, np * 4));
    if (n > 0) RC(h2d(ctx, dxy, xy, sizeof(double) * 2 * (size_t)n));
    RC(dev_laser_depth_map(L, dxy, n, dimg, W, H, fx, baseline, dout));
    RC(d2h(ctx, out, dout, np * 4));
    RC(finish(ctx));
    return L3D_OK;
    API_END(ctx)
}

int l3d_colour_mask(l3d_ctx* ctx, const uint8_t* bgr, int W, int H, const int* hsv_lo, const int* hsv_hi, int bright_thr,
                    uint8_t* mask) {
    API_BEGIN(ctx)
    NEED(ctx, bgr && hsv_lo && hsv_hi && mask && W > 0 && H > 0, "colour_mask arguments");
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = ctx->lane;
    const size_t np = (size_t)W * H;
    uint8_t* s = L.get<uint8_t>(S_SRC_L, np * 3);
    uint8_t* m = L.get<uint8_t>(S_IO_A, np);
    RC(h2d(ctx, s, bgr, np * 3));
    RC(dev_colour_mask(L, s, W, H, hsv_lo, hsv_hi, bright_thr, m));
    RC(d2h(ctx, mask, m, np));
    RC(finish(ctx));
    return L3D_OK;
    API_END(ctx)
}

// ---- raw helpers ---------------------------------------------------------------------------
void* l3d_host_alloc(long bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, (size_t)bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void l3d_host_free(void* p) { if (p) cudaFreeHost(p); }
void* l3d_dev_alloc(l3d_ctx* ctx, long bytes) {
    if (!ctx) return nullptr;
    cudaSetDevice(ctx->device);
    void* p = nullptr;
    if (cudaMalloc(&p, (size_t)bytes) != cudaSuccess) { set_err(&ctx->err, "cudaMalloc(%ld) failed", bytes); cudaGetLastError(); return nullptr; }
    return p;
}
void l3d_dev_free(l3d_ctx* ctx, void* p) { if (ctx && p) { cudaSetDevice(ctx->device); cudaFree(p); } }
int l3d_memcpy_h2d(l3d_ctx* ctx, void* dst_dev, const void* src, long bytes) {
    if (!ctx) return L3D_ERR_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemcpy(dst_dev, src, (size_t)bytes, cudaMemcpyHostToDevice));
    return L3D_OK;
}
int l3d_memcpy_d2h(l3d_ctx* ctx, void* dst, const void* src_dev, long bytes) {
    if (!ctx) return L3D_ERR_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemcpy(dst, src_dev, (size_t)bytes, cudaMemcpyDeviceToHost));
    return L3D_OK;
}

}  // extern "C"
