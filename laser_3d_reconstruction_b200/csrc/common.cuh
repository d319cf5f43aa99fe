// common.cuh -- context, lanes (stream + grow-only scratch), launch bookkeeping.
// Internal to libl3d.so; the public surface is include/l3d.h.
#pragma once
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/l3d.h"

namespace l3d {

constexpr int NUM_SMS = 148;  // B200: 2 dies x 74 SMs

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

// scratch slots (per lane)
enum Slot {
    S_SRC_L, S_SRC_R, S_RECT_L, S_RECT_R, S_GRAY_L, S_GRAY_R,
    S_DESC_L, S_DESC_R, S_COST, S_AGGR, S_DISP2, S_RAW, S_COST2, S_AGGR2, S_DISP22, S_RAW2, S_DISP_L, S_DISP_R, S_DISP_F, S_MED,
    S_LABEL, S_CNT, S_DEPTH,
    S_WLS_A, S_WLS_B, S_WLS_C, S_WLS_D, S_WLS_E, S_WLS_F, S_WLS_G, S_WLS_H, S_WLS_I, S_WLS_J, S_WLS_K,
    S_ST_GRAY, S_ST_TMP, S_ST_SM, S_ST_ROW, S_ST_CNT, S_ST_XY, S_ST_N,
    S_SM_MASK0, S_SM_MASK1, S_SM_LABEL, S_SM_LABEL2, S_SM_AREA, S_SM_ROW, S_SM_XY,
    S_RC_XY, S_RC_XYZ, S_RC_N, S_IO_A, S_IO_B, S_IO_C, S_IO_D, S_IO_E,
    S_SRC_CAP,  // frame pipeline: one staged stereo capture (both views)
    S_NUM
};

struct TimerRec {
    cudaEvent_t a, b;
};

// One stream with its own scratch: the unit of frame-level concurrency.
struct Lane {
    cudaStream_t stream = nullptr;
    cudaStream_t back_stream = nullptr;  // grouped frame pipeline: the frame's back half runs here (own priority)
    cudaEvent_t back_done = nullptr;
    DevBuf bufs[S_NUM];
    long long launches = 0;
    std::string* err = nullptr;
    unsigned* flags = nullptr;    // device word the owner (context / pipeline) provides: bit 0 = a cost volume left the int16 domain
    double wls_lut_sigma = -1.0;  // sigma_color the S_WLS_K table was built for
    // optional kernel-group timing (bench roofline leg)
    bool timing = false;
    std::map<std::string, std::vector<TimerRec>> timers;
    std::vector<cudaEvent_t> ev_pool;
    size_t ev_used = 0;

    void* get(Slot s, size_t bytes);
    template <typename T>
    T* get(Slot s, size_t count) { return (T*)get(s, count * sizeof(T)); }
    void release();
    cudaEvent_t new_event();
    void t_begin(const char* name);
    void t_end(const char* name);
    void t_reset();
};

void set_err(std::string* err, const char* fmt, ...);

#define L3D_CHECK(lane, call)                                                              \
    do {                                                                                   \
        cudaError_t e__ = (call);                                                          \
        if (e__ != cudaSuccess) {                                                          \
            l3d::set_err((lane).err, "%s:%d: %s -> %s", __FILE__, __LINE__, #call,          \
                         cudaGetErrorString(e__));                                         \
            return L3D_ERR_CUDA;                                                           \
        }                                                                                  \
    } while (0)

// L3D_DEBUG_SKIP="fgs_lines,sgbm_cost,...": launches whose kernel name contains one of the comma-separated
// substrings are skipped (results are then garbage) -- measures a kernel's marginal cost in the frame pipeline
inline bool dbg_skip(const char* kern) {
    static const char* env = getenv("L3D_DEBUG_SKIP");
    if (!env) return false;
    const char* p = env;
    while (*p) {
        const char* q = strchr(p, ',');
        size_t n = q ? (size_t)(q - p) : strlen(p);
        if (n > 0 && n < 64) {
            char tok[64];
            memcpy(tok, p, n); tok[n] = 0;
            if (strstr(kern, tok)) return true;
        }
        if (!q) break;
        p = q + 1;
    }
    return false;
}

#define L3D_LAUNCH(lane, kern, grid, block, smem, ...)                                     \
    do {                                                                                   \
        if (l3d::dbg_skip(#kern)) break;                                                   \
        kern<<<(grid), (block), (smem), (lane).stream>>>(__VA_ARGS__);                     \
        (lane).launches++;                                                                 \
        cudaError_t e__ = cudaGetLastError();                                              \
        if (e__ != cudaSuccess) {                                                          \
            l3d::set_err((lane).err, "%s:%d: launch %s -> %s", __FILE__, __LINE__, #kern,   \
                         cudaGetErrorString(e__));                                         \
            return L3D_ERR_CUDA;                                                           \
        }                                                                                  \
    } while (0)

#define L3D_ARG(lane, cond, msg)                                                           \
    do {                                                                                   \
        if (!(cond)) {                                                                     \
            l3d::set_err((lane).err, "invalid argument: %s (%s)", msg, #cond);             \
            return L3D_ERR_ARG;                                                            \
        }                                                                                  \
    } while (0)

static inline int cdiv(long a, long b) { return (int)((a + b - 1) / b); }

// fixed-point rectification map of one eye: per pixel {ix | iy<<16, ax | ay<<8}
struct RectMap {
    int2* map = nullptr;
    int W = 0, H = 0;
};

// ---- device-level stage entry points (all pointers are device pointers) -------------------
int dev_build_rectmap(Lane& L, const float* mapx_dev, const float* mapy_dev, int W, int H, int2* out);
int dev_remap_gray(Lane& L, const RectMap& m, const uint8_t* src, int sw, int sh, long stride,
                   uint8_t* rect, uint8_t* gray);
int dev_init_undistort_map(Lane& L, const double* K, const double* dist, int ndist, const double* iR, int W, int H,
                           float* mapx, float* mapy);
int dev_copy_gray(Lane& L, const uint8_t* src, int W, int H, long stride, uint8_t* bgr, uint8_t* gray);

struct SgbmDebug {
    int16_t* raw = nullptr;  // device, W*H
    int16_t* C = nullptr;    // device, HV*width1*D
    int16_t* S = nullptr;
};
int sgbm_volume_rows(const l3d_sgbm_params& p, int W, int H);
int dev_sgbm(Lane& L, const l3d_sgbm_params& p, const uint8_t* left, const uint8_t* right, int W,
             int H, int16_t* disp, SgbmDebug* dbg);
// cluster-fused aggregation of the three previous-row paths of one pass (sgbm_vgroup.cu)
bool vgroup_supported(int width1, int H, int D);
// per-job WTA outputs when a pass is the last one (nullptr array: S is written back instead)
struct VGroupWta { int16_t* raw; unsigned* d2; int W, minD, minX1, uniq; uint2* rec = nullptr; };
int dev_sgbm_vgroup(Lane& L, const int16_t* const* C, int16_t* const* S, int njobs, int width1, int H, int D, int P1,
                    int P2, int dir, const VGroupWta* wta);
// four paths per pass as a warp-skewed wavefront (sgbm_vwave.cu): wta == nullptr first pass (S written), else last pass
bool vwave_supported(int width1, int H, int D);
bool vwave_pays(int width1, int H, int D);  // ... and is it the faster choice there (measured)
int dev_sgbm_vwave(Lane& L, const int16_t* const* C, int16_t* const* S, int njobs, int width1, int H, int D, int P1,
                   int P2, int dir, const VGroupWta* wta);
int dev_voxel_downsample(Lane& L, const double* pts, int n, double voxel, int f32, double* out, int* nvox_host);
int dev_outlier_removal(Lane& L, const double* pts, int n, int nb_neighbors, double std_ratio, double* out, int* nout_host);
int dev_bm(Lane& L, const l3d_bm_params& p, const uint8_t* left, const uint8_t* right, int W, int H, int16_t* disp);
int dev_median3(Lane& L, const int16_t* src, int W, int H, int16_t* dst);
int dev_speckles(Lane& L, int16_t* img, int W, int H, int newVal, int maxSize, int maxDiff);

// depth != nullptr: the last kernel of the filter also writes the depth of the filtered disparity (dev_depth's arithmetic)
int dev_wls(Lane& L, const l3d_wls_params& p, const int16_t* dl, const int16_t* dr,
            const uint8_t* guide, int W, int H, int16_t* out, float* conf_out, float* depth = nullptr, const double* Q = nullptr);
// the FGS passes of dev_wls: `iters` x (row solves weighted by ch, column solves weighted by cv) on num/den in place
int dev_fgs(Lane& L, int solver, int variant, double lambda, int iters, const float* ch, const float* cv, int w, int h,
            float* num, float* den, float* Dscr, bool* parallel_used);
int dev_depth(Lane& L, const int16_t* disp16, int W, int H, const double* Q, float* depth);

int dev_simple(Lane& L, const uint8_t* bgr, int W, int H, const int* lo, const int* hi, int thr,
               double min_area, uint8_t* mask_morph, uint8_t* mask_final, double* xy, int* n_dev);
int dev_steger(Lane& L, const l3d_steger_params& p, const uint8_t* img, int channels, int W, int H,
               float* xy, int cap, int* n_dev);
int dev_colour_mask(Lane& L, const uint8_t* bgr, int W, int H, const int* lo, const int* hi, int thr, uint8_t* mask255);
int dev_laser_depth_map(Lane& L, const double* xy, int n, const float* disp, int W, int H, double fx, double baseline,
                        float* out);
// img: f32 depth / disparity map, or (DISPARITY kinds only) the matcher's int16 x16 disparity
template <typename T>
int dev_recon(Lane& L, const l3d_recon_params& p, const double* xy, const float* xy_f32,
              const int* n_dev, int n_max, const T* img, int W, int H, double* xyz, int* n_out_dev);
// DISPARITY_MEDIAN window: odd, 1..9 (the kernel's 81-entry sort buffer)
inline bool recon_window_ok(int window) { return window >= 1 && window <= 9 && (window & 1); }

}  // namespace l3d

namespace l3d { class HostStager; }
struct l3d_ctx {
    int device = 0;
    l3d::HostStager* stager = nullptr;  // staged host <-> device copies of the single-frame calls (hostcopy.cuh)
    unsigned* flags_host = nullptr;  // pinned mirror of lane.flags
    std::string err;
    l3d::Lane lane;
    l3d::RectMap maps[2];
};
