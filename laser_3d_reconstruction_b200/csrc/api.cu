// api.cu -- the C ABI of include/l3d.h: context, host<->device marshalling, frame pipeline.
#include <chrono>
#include <stdexcept>

#include <nvtx3/nvToolsExt.h>

#include "sgbm.cuh"
#include "hostcopy.cuh"

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

}  // namespace l3d

using namespace l3d;

#define API_BEGIN(ctxp)                                                                    \
    if (!(ctxp)) return L3D_ERR_ARG;                                                       \
    (ctxp)->stager->begin();                                                               \
    try {
#define API_END(ctxp)                                                                      \
    } catch (const std::exception& ex) {                                                   \
        (ctxp)->err = ex.what();                                                           \
        return L3D_ERR_CUDA;                                                               \
    }

#define CK(ctxp, call)                                                                     \
    do {                                                                                   \
        cudaError_t e__ = (call);                                                          \
        if (e__ != cudaSuccess) {                                                          \
            set_err(&(ctxp)->err, "%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            return L3D_ERR_CUDA;                                                           \
        }                                                                                  \
    } while (0)
#define RC(call) do { int rc__ = (call); if (rc__ != L3D_OK) return rc__; } while (0)

// Device-side domain checks of the work that just finished on `flags` (stream already synchronised).  Bit 0: a cost
// volume value reached 32768 -- OpenCV's int16 volume wraps there and this library's unsigned 16-bit arithmetic does
// not, so the result would differ from cv2 silently; reported instead (only blockSize >= 11 with P2 near its maximum
// can get there, and only on blocks whose every pixel mismatches by more than 92 % of the maximum cost).
static int check_flags(l3d_ctx* ctx, unsigned* flags) {
    if (!flags) return L3D_OK;
    unsigned h = 0;
    if (cudaMemcpy(&h, flags, sizeof(unsigned), cudaMemcpyDeviceToHost) != cudaSuccess) { cudaGetLastError(); return L3D_OK; }
    if (!h) return L3D_OK;
    cudaMemset(flags, 0, sizeof(unsigned));
    set_err(&ctx->err, "StereoSGBM: the cost volume left the int16 value domain (block sum + P2 >= 32768); cv2 wraps there, "
                       "this input is not supported");
    return L3D_ERR_UNSUPPORTED;
}
#define NEED(ctxp, cond, msg) do { if (!(cond)) { set_err(&(ctxp)->err, "invalid argument: %s", msg); return L3D_ERR_ARG; } } while (0)

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
static int set_maps(l3d_ctx* ctx, Lane& L, RectMap& m, const float* mapx, const float* mapy, int W, int H) {
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
        int minD = p->minDisparity, D = p->numDisparities;
        int width1 = (W + std::min(minD, 0)) - std::max(minD + D, 0);
        nvol = width1 > 0 ? (size_t)hv * width1 * D : 0;
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

__global__ void fill_pattern_kernel(uint32_t* p, size_t n, uint32_t seed) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, st = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += st) {
        uint32_t h = (uint32_t)i * 2654435761u + seed;
        h ^= h >> 15;
        p[i] = ((h & 0x3ffu) + 8000u) | ((((h >> 10) & 0x3ffu) + 8000u) << 16);  // plausible cost values
    }
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

int l3d_sgbm_vgroup_time(l3d_ctx* ctx, int width1, int H, int D, int P1, int P2, int njobs, int dir, int reps,
                         float* ms_per_launch) {
    API_BEGIN(ctx)
    NEED(ctx, ms_per_launch && njobs >= 1 && njobs <= 64 && reps >= 1, "vgroup_time arguments");
    NEED(ctx, vgroup_supported(width1, H, D), "geometry not supported by the cluster kernel");
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = ctx->lane;
    const size_t nvol = (size_t)width1 * H * D;
    int16_t* Cs = nullptr;
    int16_t* Ss = nullptr;
    CK(ctx, cudaMalloc(&Cs, nvol * 2 * njobs));
    if (cudaMalloc(&Ss, nvol * 2 * njobs) != cudaSuccess) { cudaFree(Cs); set_err(&ctx->err, "out of memory"); return L3D_ERR_CUDA; }
    fill_pattern_kernel<<<1024, 256, 0, L.stream>>>((uint32_t*)Cs, nvol * njobs / 2, 1u);
    cudaMemsetAsync(Ss, 0, nvol * 2 * njobs, L.stream);
    std::vector<const int16_t*> Cp(njobs);
    std::vector<int16_t*> Sp(njobs);
    for (int j = 0; j < njobs; j++) { Cp[j] = Cs + nvol * j; Sp[j] = Ss + nvol * j; }
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    int rc = dev_sgbm_vgroup(L, Cp.data(), Sp.data(), njobs, width1, H, D, P1, P2, dir, nullptr);  // warm-up
    cudaEventRecord(e0, L.stream);
    for (int r = 0; r < reps && rc == L3D_OK; r++) rc = dev_sgbm_vgroup(L, Cp.data(), Sp.data(), njobs, width1, H, D, P1, P2, dir, nullptr);
    cudaEventRecord(e1, L.stream);
    cudaError_t e = cudaEventSynchronize(e1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(Cs); cudaFree(Ss);
    if (rc != L3D_OK) return rc;
    if (e != cudaSuccess) { set_err(&ctx->err, "vgroup_time: %s", cudaGetErrorString(e)); return L3D_ERR_CUDA; }
    *ms_per_launch = ms / reps;
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

// The same path split around the cluster-fused aggregation, for the grouped frame pipeline:
// front = rectify + gray + BT operands + both matchers' cost volumes and horizontal paths;
// back  = WTA / LR check / median / speckles of both matchers + WLS + depth.
struct DepthRuns {
    SgbmRun left, right;
    bool has_right = false;
    bool vwave = false;  // the grouped pipeline aggregates this frame's volumes with the wavefront kernel
};
static int depth_front(Lane& L, const l3d_depth_config& cfg, const RectMap* maps, const uint8_t* lsrc,
                       const uint8_t* rsrc, int W, int H, long stride, uint8_t* rectL, DepthRuns& dr) {
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
static int depth_back(Lane& L, const l3d_depth_config& cfg, DepthRuns& dr, int W, int H, float* depth, int16_t* disp_f) {
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

// get_frames() depth path on device buffers (camera/single_usb_stereo_camera.py:311-359), one frame start to finish
// on its lane: the previous-row paths run direction-split (a lone volume would occupy 8 SMs in the cluster kernel)
static int depth_path(Lane& L, const l3d_depth_config& cfg, const RectMap* maps, const uint8_t* lsrc,
                      const uint8_t* rsrc, int W, int H, long stride, uint8_t* rectL, float* depth, int16_t* disp_f) {
    DepthRuns dr;
    RC(depth_front(L, cfg, maps, lsrc, rsrc, W, H, stride, rectL, dr));
    RC(sgbm_middle_split(L, dr.left, false));
    if (dr.has_right) RC(sgbm_middle_split(L, dr.right, false));
    return depth_back(L, cfg, dr, W, H, depth, disp_f);
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
    // depth_path() with the rectified view sent back as soon as it exists: its DMA and the copy into the caller's array
    // run under the matchers
    DepthRuns dr;
    RC(depth_front(L, *cfg, ctx->maps, sl, sr, W, H, stride, rl, dr));
    if (left_rect) RC(d2h(ctx, left_rect, rl, n * 3));
    RC(sgbm_middle_split(L, dr.left, false));
    if (dr.has_right) RC(sgbm_middle_split(L, dr.right, false));
    RC(depth_back(L, *cfg, dr, W, H, dp, df));
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

// ============================================================================================
// frame pipeline: nframes independent frames over `lanes` streams
// ============================================================================================
struct FrameOut {
    uint8_t* rect = nullptr; float* depth = nullptr; int16_t* disp = nullptr;
    float* xy = nullptr; double* xy64 = nullptr; double* xyz = nullptr; int* n_xy = nullptr; int* n_xyz = nullptr;
};

struct l3d_pipeline {
    l3d_ctx* ctx = nullptr;
    l3d_pipeline_config cfg;
    std::vector<Lane> lanes;
    RectMap maps[2];
    std::vector<FrameOut> outs;   // per frame slot
    void* arena = nullptr; size_t arena_cap = 0;
    int* counts_host = nullptr;   // pinned, 2*nframes
    unsigned* flags = nullptr;    // device word shared by all lanes (domain checks, see check_flags)
    int counts_cap = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::vector<cudaEvent_t> lane_done;
    cudaStream_t main = nullptr;
    float last_ms = 0.f;
    int last_frames = 0;
    // grouped mode: the frames of a lane set run their SGBM fronts on their lanes, ONE cluster-fused
    // aggregation launch per pass over all their volumes on the set's middle stream, then their backs
    static constexpr int MAXSETS = 8;
    Lane mid[MAXSETS];
    cudaEvent_t ev_mid[MAXSETS] = {};
    std::vector<cudaEvent_t> lane_front;
    std::vector<DepthRuns> runs;  // per lane
    bool timing = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> dbg_events;
    // Steady-state replay: a step with the same buffers and frame count as the previous one is captured once
    // (all lane / aggregation / back streams fork from and join `main`) and replayed as a CUDA graph -- the
    // 34 launches per frame otherwise make small configurations (320x360) host-launch-bound.
    struct GraphKey {
        const void *left, *right, *depth_h, *xyz_h; int nframes; bool host_in;
        bool operator==(const GraphKey& o) const {
            return left == o.left && right == o.right && depth_h == o.depth_h && xyz_h == o.xyz_h && nframes == o.nframes && host_in == o.host_in;
        }
    };
    struct GraphEntry { GraphKey key; int seen = 0; bool launch_bound = false; cudaGraphExec_t exec = nullptr; long long launches = 0; };
    std::vector<GraphEntry> graphs;
    bool graphs_ok = true;          // cleared when a capture fails: the pipeline then stays on direct launches
    long long graph_launches = 0;   // kernel launches performed by graph replays
    long long graph_replays = 0;
    cudaEvent_t ev_fork = nullptr;
    // L3D_DEBUG_PHASES: tagged timeline marks (tag, frame, event) printed relative to the run's first enqueue
    struct Mark { const char* tag; int frame; cudaEvent_t ev; };
    std::vector<Mark> dbg_marks;
    void mark(const char* tag, int frame, cudaStream_t s) {
        cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, s); dbg_marks.push_back({tag, frame, e});
    }
};

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// captured graphs hold raw device / pinned pointers: drop them whenever one of those buffers is reallocated
static void pipe_drop_graphs(l3d_pipeline* p) {
    for (auto& g : p->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
    p->graphs.clear();
}

static int pipe_prepare(l3d_pipeline* p, int nframes) {
    l3d_ctx* ctx = p->ctx;
    const int W = p->cfg.W, H = p->cfg.H, cap = p->cfg.max_points;
    size_t n = (size_t)W * H;
    size_t per = align_up(n * 3, 256) + align_up(n * 4, 256) + align_up(n * 2, 256) + align_up((size_t)cap * 8, 256) +
                 align_up((size_t)cap * 16, 256) + align_up((size_t)cap * 24, 256) + 512;
    size_t need = per * nframes;
    if (need > p->arena_cap) {
        pipe_drop_graphs(p);
        for (auto& L : p->lanes) CK(ctx, cudaStreamSynchronize(L.stream));
        if (p->arena) cudaFree(p->arena);
        p->arena = nullptr; p->arena_cap = 0;
        CK(ctx, cudaMalloc(&p->arena, need));
        p->arena_cap = need;
        p->outs.clear();
    }
    if ((int)p->outs.size() < nframes) {
        p->outs.resize(nframes);
        char* base = (char*)p->arena;
        for (int f = 0; f < nframes; f++) {
            char* q = base + per * f;
            FrameOut& o = p->outs[f];
            o.rect = (uint8_t*)q; q += align_up(n * 3, 256);
            o.depth = (float*)q; q += align_up(n * 4, 256);
            o.disp = (int16_t*)q; q += align_up(n * 2, 256);
            o.xy = (float*)q; q += align_up((size_t)cap * 8, 256);
            o.xy64 = (double*)q; q += align_up((size_t)cap * 16, 256);
            o.xyz = (double*)q; q += align_up((size_t)cap * 24, 256);
            o.n_xy = (int*)q; o.n_xyz = (int*)(q + 256);
        }
    }
    if (p->counts_cap < nframes) {
        pipe_drop_graphs(p);
        if (p->counts_host) cudaFreeHost(p->counts_host);
        CK(ctx, cudaMallocHost(&p->counts_host, sizeof(int) * 2 * (size_t)nframes));
        p->counts_cap = nframes;
    }
    return L3D_OK;
}

// enqueue one frame on lane L (all device pointers)
static int pipe_extract(l3d_pipeline* p, Lane& L, FrameOut& o);
static int pipe_frame(l3d_pipeline* p, Lane& L, const uint8_t* l, const uint8_t* r, FrameOut& o) {
    const l3d_pipeline_config& c = p->cfg;
    RC(depth_path(L, c.depth, p->maps, l, r, c.W, c.H, 3L * c.W, o.rect, o.depth, o.disp));
    return pipe_extract(p, L, o);
}
// laser centre line on the rectified left image + 3D points (main.py:172-178)
static int pipe_extract(l3d_pipeline* p, Lane& L, FrameOut& o) {
    const l3d_pipeline_config& c = p->cfg;
    const int W = c.W, H = c.H;
    if (c.extractor < 0) {
        L3D_CHECK(L, cudaMemsetAsync(o.n_xy, 0, sizeof(int), L.stream));
        L3D_CHECK(L, cudaMemsetAsync(o.n_xyz, 0, sizeof(int), L.stream));
        return L3D_OK;
    }
    const double* xy64 = nullptr; const float* xy32 = nullptr;
    L.t_begin("extract");
    if (c.extractor == 4) {
        RC(dev_simple(L, o.rect, W, H, c.simple_hsv_lo, c.simple_hsv_hi, c.simple_bright_thr, c.simple_min_area,
                      nullptr, nullptr, o.xy64, o.n_xy));
        xy64 = o.xy64;
    } else {
        RC(dev_steger(L, c.steger, o.rect, 3, W, H, o.xy, c.max_points, o.n_xy));
        xy32 = o.xy;
    }
    L.t_end("extract");
    const float* img = (c.recon.kind == L3D_RECON_PLANE) ? nullptr : o.depth;
    L.t_begin("recon");
    RC(dev_recon(L, c.recon, xy64, xy32, o.n_xy, c.max_points, img, W, H, o.xyz, o.n_xyz));
    L.t_end("recon");
    return L3D_OK;
}

// rows (frame_id, x, y, z) of up to PACK_FRAMES frames per launch
constexpr int PACK_FRAMES = 64;
struct PackArgs {
    const double* xyz[PACK_FRAMES];
    long long off[PACK_FRAMES];
    int cnt[PACK_FRAMES], fid[PACK_FRAMES];
    int n;
};
__global__ void pack_points_kernel(const PackArgs a, double* __restrict__ table) {
    const int f = blockIdx.y;
    if (f >= a.n) return;
    const double* src = a.xyz[f];
    double* dst = table + a.off[f] * 4;
    const double id = (double)a.fid[f];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < a.cnt[f]; i += gridDim.x * blockDim.x) {
        dst[4 * (size_t)i] = id;
        dst[4 * (size_t)i + 1] = src[3 * (size_t)i];
        dst[4 * (size_t)i + 2] = src[3 * (size_t)i + 1];
        dst[4 * (size_t)i + 3] = src[3 * (size_t)i + 2];
    }
}

extern "C" {

int l3d_pipeline_pack_points_dev(l3d_pipeline* p, int nframes, const int* frame_ids, double* table_dev,
                                 long long* total_rows) {
    if (!p) return L3D_ERR_ARG;
    l3d_ctx* ctx = p->ctx;
    API_BEGIN(ctx)
    NEED(ctx, nframes >= 0 && nframes <= p->last_frames && frame_ids && total_rows, "pack_points arguments");
    CK(ctx, cudaSetDevice(ctx->device));
    Lane& L = p->lanes[0];
    long long off = 0;
    for (int f0 = 0; f0 < nframes; f0 += PACK_FRAMES) {
        PackArgs a;
        a.n = std::min(PACK_FRAMES, nframes - f0);
        int maxc = 0;
        for (int i = 0; i < a.n; i++) {
            const int f = f0 + i;
            a.xyz[i] = p->outs[f].xyz; a.cnt[i] = p->counts_host[2 * f + 1]; a.fid[i] = frame_ids[f]; a.off[i] = off;
            off += a.cnt[i];
            maxc = std::max(maxc, a.cnt[i]);
        }
        if (maxc > 0) {
            NEED(ctx, table_dev, "pack_points table");
            L3D_LAUNCH(L, pack_points_kernel, dim3(std::max(1, std::min(cdiv(maxc, 256), 64)), a.n), 256, 0, a, table_dev);
        }
    }
    CK(ctx, cudaStreamSynchronize(L.stream));
    *total_rows = off;
    return L3D_OK;
    API_END(ctx)
}

int l3d_pipeline_create(l3d_ctx* ctx, const l3d_pipeline_config* cfg, l3d_pipeline** out) {
    API_BEGIN(ctx)
    NEED(ctx, cfg && out, "pipeline_create arguments");
    NEED(ctx, cfg->W > 1 && cfg->H > 0 && cfg->lanes >= 1 && cfg->lanes <= 64 && cfg->max_points > 0, "pipeline config");
    NEED(ctx, cfg->extractor >= -1 && cfg->extractor <= 4, "pipeline extractor");
    if (cfg->extractor == 4) NEED(ctx, cfg->max_points >= cfg->H, "max_points must be >= H for the Simple extractor");
    CK(ctx, cudaSetDevice(ctx->device));
    l3d_pipeline* p = new l3d_pipeline();
    p->ctx = ctx; p->cfg = *cfg;
    p->lanes.resize(cfg->lanes);
    // Stream priorities.  The cluster-fused aggregation needs 8 completely free SMs of one GPC per volume, so its
    // launches go first whenever they are ready (any resident CTA of another kernel blocks a cluster CTA: it takes
    // the whole register file); the short back-half kernels come next, the wide front kernels fill the rest.
    int prio_lo = 0, prio_hi = 0;
    CK(ctx, cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    int prio[3] = {prio_hi, prio_lo, std::max(prio_hi, prio_lo - 2)};  // aggregation, front, back
    if (const char* e = getenv("L3D_PRIO")) sscanf(e, "%d,%d,%d", &prio[0], &prio[1], &prio[2]);
    for (int& q : prio) q = std::min(prio_lo, std::max(prio_hi, q));
    CK(ctx, cudaMalloc(&p->flags, 16));
    CK(ctx, cudaMemset(p->flags, 0, 16));
    for (auto& L : p->lanes) {
        L.err = &ctx->err;
        L.flags = p->flags;
        CK(ctx, cudaStreamCreateWithPriority(&L.stream, cudaStreamNonBlocking, prio[1]));
        CK(ctx, cudaStreamCreateWithPriority(&L.back_stream, cudaStreamNonBlocking, prio[2]));
        CK(ctx, cudaEventCreateWithFlags(&L.back_done, cudaEventDisableTiming));
    }
    CK(ctx, cudaStreamCreateWithFlags(&p->main, cudaStreamNonBlocking));
    CK(ctx, cudaEventCreate(&p->ev0));
    CK(ctx, cudaEventCreate(&p->ev1));
    CK(ctx, cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming));
    p->lane_done.resize(cfg->lanes);
    for (auto& e : p->lane_done) CK(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    p->lane_front.resize(cfg->lanes);
    for (auto& e : p->lane_front) CK(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    p->runs.resize(cfg->lanes);
    for (int i = 0; i < l3d_pipeline::MAXSETS; i++) {
        p->mid[i].err = &ctx->err;
        p->mid[i].flags = p->flags;
        CK(ctx, cudaStreamCreateWithPriority(&p->mid[i].stream, cudaStreamNonBlocking, prio[0]));
        CK(ctx, cudaEventCreateWithFlags(&p->ev_mid[i], cudaEventDisableTiming));
    }
    *out = p;
    return L3D_OK;
    API_END(ctx)
}

void l3d_pipeline_destroy(l3d_pipeline* p) {
    if (!p) return;
    cudaSetDevice(p->ctx->device);
    for (auto& L : p->lanes) L.release();
    for (int i = 0; i < l3d_pipeline::MAXSETS; i++) { p->mid[i].release(); if (p->ev_mid[i]) cudaEventDestroy(p->ev_mid[i]); }
    for (auto e : p->lane_front) cudaEventDestroy(e);
    for (auto& m : p->maps) if (m.map) cudaFree(m.map);
    if (p->arena) cudaFree(p->arena);
    if (p->flags) cudaFree(p->flags);
    if (p->counts_host) cudaFreeHost(p->counts_host);
    pipe_drop_graphs(p);
    if (p->ev0) cudaEventDestroy(p->ev0);
    if (p->ev1) cudaEventDestroy(p->ev1);
    if (p->ev_fork) cudaEventDestroy(p->ev_fork);
    for (auto e : p->lane_done) cudaEventDestroy(e);
    if (p->main) cudaStreamDestroy(p->main);
    delete p;
}

int l3d_pipeline_set_maps(l3d_pipeline* p, int eye, const float* mapx, const float* mapy) {
    if (!p) return L3D_ERR_ARG;
    l3d_ctx* ctx = p->ctx;
    API_BEGIN(ctx)
    NEED(ctx, (eye == 0 || eye == 1) && mapx && mapy, "pipeline_set_maps arguments");
    CK(ctx, cudaSetDevice(ctx->device));
    pipe_drop_graphs(p);
    return set_maps(ctx, p->lanes[0], p->maps[eye], mapx, mapy, p->cfg.W, p->cfg.H);
    API_END(ctx)
}

// Grouped mode: one aggregation launch should carry close to (but not more than) one wave of clusters --
// 15 clusters of 8 CTAs (14 of 9) are resident on a B200 (cudaOccupancyMaxActiveClusters) -- so a lane set is
// 7 frames with WLS (14 volumes) or 15 without; up to 4 sets alternate to overlap fronts/backs with
// another set's aggregation.
constexpr int VG_WAVE = 15;
static int pipe_group_size(const l3d_pipeline* p) {
    const int jobs_per_frame = p->cfg.depth.use_wls ? 2 : 1;
    static const int forced = getenv("L3D_GROUP") ? atoi(getenv("L3D_GROUP")) : 0;  // experiment: frames per lane set
    if (forced > 0) return std::min((int)p->lanes.size(), forced);
    return std::min((int)p->lanes.size(), std::max(1, VG_WAVE / jobs_per_frame));
}
static bool pipe_grouped(const l3d_pipeline* p) {
    static const bool off = getenv("L3D_NO_VGROUP") && atoi(getenv("L3D_NO_VGROUP")) > 0;
    if (off) return false;
    const l3d_pipeline_config& c = p->cfg;
    const int jobs_per_frame = c.depth.use_wls ? 2 : 1;
    if (pipe_group_size(p) * jobs_per_frame < 8 || c.depth.left.mode >= 2) return false;  // 3WAY / HH4: direction-split
    const l3d_sgbm_params& q = c.depth.left;
    const int width1 = (c.W + std::min(q.minDisparity, 0)) - std::max(q.minDisparity + q.numDisparities, 0);
    return width1 > 0 && vgroup_supported(width1, c.H, q.numDisparities);
}

static int pipe_run_grouped(l3d_pipeline* p, const uint8_t* left, const uint8_t* right, bool host_in, int nframes,
                            float* depth_h, double* xyz_h) {
    l3d_ctx* ctx = p->ctx;
    const l3d_pipeline_config& c = p->cfg;
    const int W = c.W, H = c.H, cap = c.max_points;
    const size_t nb = (size_t)W * H * 3, n = (size_t)W * H;
    const int nl = (int)p->lanes.size();
    const int gsz = pipe_group_size(p);
    const int nsets = p->timing ? 1 : std::max(1, std::min(l3d_pipeline::MAXSETS, nl / gsz));  // lane sets alternate
    const int nchunks = (nframes + gsz - 1) / gsz;
    const l3d_sgbm_params& lp = c.depth.left;
    const bool use_vwave = sgbm_vwave_ok((W + std::min(lp.minDisparity, 0)) - std::max(lp.minDisparity + lp.numDisparities, 0), H,
                                         lp.numDisparities, lp.mode);
    for (int i = 0; i < l3d_pipeline::MAXSETS; i++) {
        p->mid[i].t_reset(); p->mid[i].timing = p->timing;
        // only streams that get work: every stream that forks from `main` has to join it again (graph capture)
        if (i < std::min(nsets, nchunks)) CK(ctx, cudaStreamWaitEvent(p->mid[i].stream, p->ev_fork, 0));
    }
    int chunk = 0;
    for (int f0 = 0; f0 < nframes; f0 += gsz, chunk++) {
        const int set = chunk % nsets, ng = std::min(gsz, nframes - f0);
        Lane& M = p->mid[set];
        std::vector<SgbmRun*> list;
        for (int i = 0; i < ng; i++) {
            const int li = set * gsz + i, f = f0 + i;
            Lane& L = p->lanes[li];
            const uint8_t *l = left + nb * f, *r = right + nb * f;
            if (p->timing && i > 0) CK(ctx, cudaStreamWaitEvent(L.stream, p->lane_front[li - 1], 0));  // kernels alone
            if (host_in) {
                uint8_t* sl = L.get<uint8_t>(S_SRC_L, nb);
                uint8_t* sr = L.get<uint8_t>(S_SRC_R, nb);
                L3D_CHECK(L, cudaMemcpyAsync(sl, l, nb, cudaMemcpyHostToDevice, L.stream));
                L3D_CHECK(L, cudaMemcpyAsync(sr, r, nb, cudaMemcpyHostToDevice, L.stream));
                l = sl; r = sr;
            }
            DepthRuns& dr = p->runs[li];
            dr.vwave = use_vwave;
            static const bool dbg_marks_on = getenv("L3D_DEBUG_PHASES") != nullptr;
            if (dbg_marks_on) p->mark("front0", f, L.stream);
            RC(depth_front(L, c.depth, p->maps, l, r, W, H, 3L * W, p->outs[f].rect, dr));
            if (dbg_marks_on) p->mark("front1", f, L.stream);
            CK(ctx, cudaEventRecord(p->lane_front[li], L.stream));
            CK(ctx, cudaStreamWaitEvent(M.stream, p->lane_front[li], 0));
            list.push_back(&dr.left);
            if (dr.has_right) list.push_back(&dr.right);
        }
        static const bool dbg_phases = getenv("L3D_DEBUG_PHASES") != nullptr;
        cudaEvent_t d0 = nullptr, d1 = nullptr;
        if (dbg_phases) { cudaEventCreate(&d0); cudaEventCreate(&d1); cudaEventRecord(d0, M.stream); }
        if (use_vwave) RC(sgbm_middle_vwave(M, list.data(), (int)list.size()));
        else RC(sgbm_middle_vgroup(M, list.data(), (int)list.size(), false));
        if (dbg_phases) { cudaEventRecord(d1, M.stream); p->dbg_events.push_back({d0, d1}); }
        CK(ctx, cudaEventRecord(p->ev_mid[set], M.stream));
        for (int i = 0; i < ng; i++) {
            const int li = set * gsz + i, f = f0 + i;
            Lane& L = p->lanes[li];
            FrameOut& o = p->outs[f];
            // the back half runs on the lane's second stream (own priority); the lane's main stream rejoins below
            cudaStream_t front_stream = L.stream;
            if (!p->timing) {
                CK(ctx, cudaStreamWaitEvent(L.back_stream, p->lane_front[li], 0));
                L.stream = L.back_stream;
            }
            struct Restore { Lane& l; cudaStream_t s; ~Restore() { l.stream = s; } } restore{L, front_stream};
            CK(ctx, cudaStreamWaitEvent(L.stream, p->ev_mid[set], 0));
            if (p->timing && i > 0) CK(ctx, cudaStreamWaitEvent(L.stream, p->lane_done[li - 1], 0));
            if (dbg_phases) p->mark("back0", f, L.stream);
            RC(depth_back(L, c.depth, p->runs[li], W, H, o.depth, o.disp));
            if (dbg_phases) p->mark("back1", f, L.stream);
            RC(pipe_extract(p, L, o));
            if (dbg_phases) p->mark("extr1", f, L.stream);
            L3D_CHECK(L, cudaMemcpyAsync(p->counts_host + 2 * f, o.n_xy, sizeof(int), cudaMemcpyDeviceToHost, L.stream));
            L3D_CHECK(L, cudaMemcpyAsync(p->counts_host + 2 * f + 1, o.n_xyz, sizeof(int), cudaMemcpyDeviceToHost, L.stream));
            if (depth_h) L3D_CHECK(L, cudaMemcpyAsync(depth_h + n * f, o.depth, n * 4, cudaMemcpyDeviceToHost, L.stream));
            if (xyz_h) L3D_CHECK(L, cudaMemcpyAsync(xyz_h + (size_t)cap * 3 * f, o.xyz, (size_t)cap * 24, cudaMemcpyDeviceToHost, L.stream));
            if (p->timing) CK(ctx, cudaEventRecord(p->lane_done[li], L.stream));
            if (!p->timing) {
                CK(ctx, cudaEventRecord(L.back_done, L.back_stream));
                CK(ctx, cudaStreamWaitEvent(front_stream, L.back_done, 0));
            }
        }
    }
    return L3D_OK;
}

// fork from `main`, enqueue one step on the lanes, join `main` again (capturable: no allocation in the steady state)
static int pipe_enqueue(l3d_pipeline* p, const uint8_t* left, const uint8_t* right, bool host_in, int nframes,
                        float* depth_h, double* xyz_h) {
    l3d_ctx* ctx = p->ctx;
    const int W = p->cfg.W, H = p->cfg.H, cap = p->cfg.max_points;
    const size_t nb = (size_t)W * H * 3, n = (size_t)W * H;
    const int nl = (int)p->lanes.size();
    CK(ctx, cudaEventRecord(p->ev_fork, p->main));
    for (auto& L : p->lanes) CK(ctx, cudaStreamWaitEvent(L.stream, p->ev_fork, 0));
    const bool grouped = pipe_grouped(p);
    if (grouped) RC(pipe_run_grouped(p, left, right, host_in, nframes, depth_h, xyz_h));
    for (int f = 0; f < nframes && !grouped; f++) {
        Lane& L = p->lanes[f % nl];
        FrameOut& o = p->outs[f];
        const uint8_t *l = left + nb * f, *r = right + nb * f;
        if (host_in) {
            uint8_t* sl = L.get<uint8_t>(S_SRC_L, nb);
            uint8_t* sr = L.get<uint8_t>(S_SRC_R, nb);
            L3D_CHECK(L, cudaMemcpyAsync(sl, l, nb, cudaMemcpyHostToDevice, L.stream));
            L3D_CHECK(L, cudaMemcpyAsync(sr, r, nb, cudaMemcpyHostToDevice, L.stream));
            l = sl; r = sr;
        }
        RC(pipe_frame(p, L, l, r, o));
        L3D_CHECK(L, cudaMemcpyAsync(p->counts_host + 2 * f, o.n_xy, sizeof(int), cudaMemcpyDeviceToHost, L.stream));
        L3D_CHECK(L, cudaMemcpyAsync(p->counts_host + 2 * f + 1, o.n_xyz, sizeof(int), cudaMemcpyDeviceToHost, L.stream));
        if (depth_h) L3D_CHECK(L, cudaMemcpyAsync(depth_h + n * f, o.depth, n * 4, cudaMemcpyDeviceToHost, L.stream));
        if (xyz_h) L3D_CHECK(L, cudaMemcpyAsync(xyz_h + (size_t)cap * 3 * f, o.xyz, (size_t)cap * 24, cudaMemcpyDeviceToHost, L.stream));
    }
    for (int i = 0; i < nl; i++) {
        CK(ctx, cudaEventRecord(p->lane_done[i], p->lanes[i].stream));
        CK(ctx, cudaStreamWaitEvent(p->main, p->lane_done[i], 0));
    }
    return L3D_OK;
}

static long long pipe_launches_now(const l3d_pipeline* p) {
    long long s = 0;
    for (auto& L : p->lanes) s += L.launches;
    for (int i = 0; i < l3d_pipeline::MAXSETS; i++) s += p->mid[i].launches;
    return s;
}

static int pipe_run(l3d_pipeline* p, const uint8_t* left, const uint8_t* right, bool host_in, int nframes,
                    float* depth_h, double* xyz_h, int* counts) {
    l3d_ctx* ctx = p->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    RC(pipe_prepare(p, nframes));
    for (auto& L : p->lanes) L.t_reset();
    auto t_enq0 = std::chrono::steady_clock::now();
    // ---- CUDA-graph replay of a repeated step (same buffers, same frame count); the first occurrence runs with
    // direct launches (it also grows the scratch buffers), the second decides whether the step is launch-bound,
    // the third is captured, later ones are replayed
    static const bool graphs_off = (getenv("L3D_NO_GRAPH") && atoi(getenv("L3D_NO_GRAPH")) > 0) || getenv("L3D_DEBUG_PHASES") ||
                                   getenv("L3D_DEBUG_SKIP");
    l3d_pipeline::GraphEntry* ge = nullptr;
    if (!graphs_off && p->graphs_ok && !p->timing) {
        const l3d_pipeline::GraphKey key{left, right, depth_h, xyz_h, nframes, host_in};
        for (auto& g : p->graphs) if (g.key == key) ge = &g;
        if (!ge) {
            if (p->graphs.size() >= 8) {  // bounded cache: drop the oldest entry
                if (p->graphs.front().exec) cudaGraphExecDestroy(p->graphs.front().exec);
                p->graphs.erase(p->graphs.begin());
            }
            p->graphs.push_back(l3d_pipeline::GraphEntry());
            ge = &p->graphs.back();
            ge->key = key;
        }
        ge->seen++;
    }
    bool replayed = false;
    static const bool graphs_always = getenv("L3D_GRAPH") && atoi(getenv("L3D_GRAPH")) > 0;
    if (ge && ge->seen >= 3 && (ge->launch_bound || graphs_always)) {
        if (!ge->exec) {
            const long long l0 = pipe_launches_now(p);
            cudaGraph_t graph = nullptr;
            cudaError_t e = cudaStreamBeginCapture(p->main, cudaStreamCaptureModeRelaxed);
            int rc = L3D_OK;
            if (e == cudaSuccess) {
                rc = pipe_enqueue(p, left, right, host_in, nframes, depth_h, xyz_h);
                e = cudaStreamEndCapture(p->main, &graph);
            }
            if (e == cudaSuccess && rc == L3D_OK && graph) e = cudaGraphInstantiate(&ge->exec, graph, 0);
            if (graph) cudaGraphDestroy(graph);
            ge->launches = pipe_launches_now(p) - l0;
            // (the counters the capture incremented stand for the first replay)
            if (e != cudaSuccess || rc != L3D_OK || !ge->exec) {
                cudaGetLastError();
                p->graphs_ok = false;  // stay on direct launches
                if (ge->exec) { cudaGraphExecDestroy(ge->exec); ge->exec = nullptr; }
                if (rc != L3D_OK && e == cudaSuccess) return rc;
            } else {
                p->graph_launches -= ge->launches;  // the replay below adds them back: counted once
            }
        }
        if (ge->exec) {
            CK(ctx, cudaEventRecord(p->ev0, p->main));
            CK(ctx, cudaGraphLaunch(ge->exec, p->main));
            p->graph_launches += ge->launches;
            p->graph_replays++;
            replayed = true;
        }
    }
    if (!replayed) {
        CK(ctx, cudaEventRecord(p->ev0, p->main));
        RC(pipe_enqueue(p, left, right, host_in, nframes, depth_h, xyz_h));
    }
    CK(ctx, cudaEventRecord(p->ev1, p->main));
    const double enq_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_enq0).count();
    if (getenv("L3D_DEBUG_ENQUEUE"))
        fprintf(stderr, "[l3d] enqueue of %d frames took %.3f ms host time%s\n", nframes, enq_ms, replayed ? " (graph replay)" : "");
    CK(ctx, cudaEventSynchronize(p->ev1));
    CK(ctx, cudaEventElapsedTime(&p->last_ms, p->ev0, p->ev1));
    // a step whose direct enqueue takes a large part of its GPU time is launch-bound: replay it as a graph from now on
    // (at config 3 the enqueue is 12 % of the step and direct launches with stream priorities are 2 % faster)
    // (judged on the second occurrence: the first one also allocates the scratch buffers)
    if (ge && !replayed && ge->seen == 2) ge->launch_bound = enq_ms > 0.4 * (double)p->last_ms;
    for (auto& e : p->dbg_events) {
        float a = 0.f, b = 0.f;
        cudaEventElapsedTime(&a, p->ev0, e.first); cudaEventElapsedTime(&b, p->ev0, e.second);
        fprintf(stderr, "[l3d] aggregation launch pair: start %.2f ms, end %.2f ms (total run %.2f ms)\n", a, b, p->last_ms);
        cudaEventDestroy(e.first); cudaEventDestroy(e.second);
    }
    p->dbg_events.clear();
    for (auto& m : p->dbg_marks) {
        float a = 0.f;
        cudaEventElapsedTime(&a, p->ev0, m.ev);
        fprintf(stderr, "[l3d] mark %-7s frame %3d at %8.3f ms\n", m.tag, m.frame, a);
        cudaEventDestroy(m.ev);
    }
    p->dbg_marks.clear();
    p->last_frames = nframes;
    if (counts) for (int f = 0; f < nframes; f++) counts[f] = p->counts_host[2 * f + 1];
    return check_flags(ctx, p->flags);
}

int l3d_pipeline_run_dev(l3d_pipeline* p, const uint8_t* left_dev, const uint8_t* right_dev, int nframes, int* counts) {
    if (!p) return L3D_ERR_ARG;
    l3d_ctx* ctx = p->ctx;
    API_BEGIN(ctx)
    NEED(ctx, left_dev && right_dev && nframes > 0, "pipeline_run_dev arguments");
    return pipe_run(p, left_dev, right_dev, false, nframes, nullptr, nullptr, counts);
    API_END(ctx)
}

int l3d_pipeline_run_host(l3d_pipeline* p, const uint8_t* left, const uint8_t* right, int nframes, float* depth,
                          double* xyz, int* counts) {
    if (!p) return L3D_ERR_ARG;
    l3d_ctx* ctx = p->ctx;
    API_BEGIN(ctx)
    NEED(ctx, left && right && nframes > 0, "pipeline_run_host arguments");
    return pipe_run(p, left, right, true, nframes, depth, xyz, counts);
    API_END(ctx)
}

int l3d_pipeline_fetch(l3d_pipeline* p, int frame, uint8_t* left_rect, float* depth, int16_t* disp, float* xy,
                       double* xyz, int* n_xy, int* n_xyz) {
    if (!p) return L3D_ERR_ARG;
    l3d_ctx* ctx = p->ctx;
    API_BEGIN(ctx)
    NEED(ctx, frame >= 0 && frame < p->last_frames, "frame index");
    CK(ctx, cudaSetDevice(ctx->device));
    const FrameOut& o = p->outs[frame];
    size_t n = (size_t)p->cfg.W * p->cfg.H;
    int nxy = p->counts_host[2 * frame], nxyz = p->counts_host[2 * frame + 1];
    if (n_xy) *n_xy = nxy;
    if (n_xyz) *n_xyz = nxyz;
    if (left_rect) CK(ctx, cudaMemcpy(left_rect, o.rect, n * 3, cudaMemcpyDeviceToHost));
    if (depth) CK(ctx, cudaMemcpy(depth, o.depth, n * 4, cudaMemcpyDeviceToHost));
    if (disp) CK(ctx, cudaMemcpy(disp, o.disp, n * 2, cudaMemcpyDeviceToHost));
    int m = std::min(nxy, p->cfg.max_points);
    if (xy && m > 0) {
        if (p->cfg.extractor == 4) {
            std::vector<double> t((size_t)2 * m);
            CK(ctx, cudaMemcpy(t.data(), o.xy64, sizeof(double) * 2 * m, cudaMemcpyDeviceToHost));
            for (int i = 0; i < 2 * m; i++) xy[i] = (float)t[i];
        } else CK(ctx, cudaMemcpy(xy, o.xy, sizeof(float) * 2 * m, cudaMemcpyDeviceToHost));
    }
    if (xyz && nxyz > 0) CK(ctx, cudaMemcpy(xyz, o.xyz, sizeof(double) * 3 * nxyz, cudaMemcpyDeviceToHost));
    return L3D_OK;
    API_END(ctx)
}

int l3d_pipeline_fetch_points(l3d_pipeline* p, int frame, double* xy, int xy_cap, double* xyz, int xyz_cap, int* n_xy,
                              int* n_xyz) {
    if (!p) return L3D_ERR_ARG;
    l3d_ctx* ctx = p->ctx;
    API_BEGIN(ctx)
    NEED(ctx, frame >= 0 && frame < p->last_frames && xy_cap >= 0 && xyz_cap >= 0, "fetch_points arguments");
    CK(ctx, cudaSetDevice(ctx->device));
    const FrameOut& o = p->outs[frame];
    const int nxy = p->counts_host[2 * frame], nxyz = p->counts_host[2 * frame + 1];
    if (n_xy) *n_xy = nxy;
    if (n_xyz) *n_xyz = nxyz;
    const int m = std::min(std::min(nxy, p->cfg.max_points), xy_cap);
    if (xy && m > 0) {
        if (p->cfg.extractor == 4) {
            CK(ctx, cudaMemcpy(xy, o.xy64, sizeof(double) * 2 * m, cudaMemcpyDeviceToHost));
        } else {
            std::vector<float> t((size_t)2 * m);
            CK(ctx, cudaMemcpy(t.data(), o.xy, sizeof(float) * 2 * m, cudaMemcpyDeviceToHost));
            for (int i = 0; i < 2 * m; i++) xy[i] = (double)t[i];
        }
    }
    const int m3 = std::min(std::min(nxyz, p->cfg.max_points), xyz_cap);
    if (xyz && m3 > 0) CK(ctx, cudaMemcpy(xyz, o.xyz, sizeof(double) * 3 * m3, cudaMemcpyDeviceToHost));
    return L3D_OK;
    API_END(ctx)
}

int l3d_pipeline_points_needed(l3d_pipeline* p) {
    if (!p) return -1;
    int m = 0;
    for (int f = 0; f < p->last_frames; f++) m = std::max(m, p->counts_host[2 * f]);
    return m;
}

long long l3d_pipeline_launch_count(l3d_pipeline* p) {
    long long s = 0;
    if (p) {
        for (auto& L : p->lanes) s += L.launches;
        for (int i = 0; i < l3d_pipeline::MAXSETS; i++) s += p->mid[i].launches;
        s += p->graph_launches;
    }
    return s;
}

long long l3d_pipeline_graph_replays(l3d_pipeline* p) { return p ? p->graph_replays : 0; }

int l3d_pipeline_set_timing(l3d_pipeline* p, int on) {
    if (!p) return L3D_ERR_ARG;
    for (auto& L : p->lanes) L.timing = on != 0;
    p->timing = on != 0;  // grouped mode: lanes are chained so that every timed kernel runs alone
    return L3D_OK;
}

float l3d_pipeline_last_ms(l3d_pipeline* p) { return p ? p->last_ms : 0.f; }

int l3d_pipeline_kernel_time(l3d_pipeline* p, const char* which, float* ms, int* launches) {
    if (!p || !which || !ms || !launches) return L3D_ERR_ARG;
    l3d_ctx* ctx = p->ctx;
    float tot = 0.f; int cnt = 0;
    std::vector<Lane*> all;
    for (auto& L : p->lanes) all.push_back(&L);
    for (int i = 0; i < l3d_pipeline::MAXSETS; i++) all.push_back(&p->mid[i]);
    for (Lane* Lp : all) {
        Lane& L = *Lp;
        auto it = L.timers.find(which);
        if (it == L.timers.end()) continue;
        for (auto& r : it->second) {
            if (!r.b) continue;
            float t = 0.f;
            CK(ctx, cudaEventSynchronize(r.b));
            CK(ctx, cudaEventElapsedTime(&t, r.a, r.b));
            tot += t; cnt++;
        }
    }
    *ms = tot; *launches = cnt;
    return L3D_OK;
}

}  // extern "C"
