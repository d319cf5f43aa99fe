// api.cuh -- what the two translation units of the C ABI share: api.cu (context, single-frame calls) and pipeline.cu
// (frame pipeline).  Internal to libl3d.so.
#pragma once
#include "sgbm.cuh"
#include "hostcopy.cuh"

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
            l3d::set_err(&(ctxp)->err, "%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            return L3D_ERR_CUDA;                                                           \
        }                                                                                  \
    } while (0)
#define RC(call) do { int rc__ = (call); if (rc__ != L3D_OK) return rc__; } while (0)
#define NEED(ctxp, cond, msg) do { if (!(cond)) { l3d::set_err(&(ctxp)->err, "invalid argument: %s", msg); return L3D_ERR_ARG; } } while (0)

namespace l3d {

// Device-side domain checks of the work that just finished on `flags` (stream already synchronised).  Bit 0: a cost
// volume value reached 32768 -- OpenCV's int16 volume wraps there and this library's unsigned 16-bit arithmetic does
// not, so the result would differ from cv2 silently; reported instead (only blockSize >= 11 with P2 near its maximum
// can get there, and only on blocks whose every pixel mismatches by more than 92 % of the maximum cost).
int check_flags(l3d_ctx* ctx, unsigned* flags);
// upload one eye's cv2 maps and build its fixed-point map on L (synchronises L)
int set_maps(l3d_ctx* ctx, Lane& L, RectMap& m, const float* mapx, const float* mapy, int W, int H);

// get_frames()'s depth path on device buffers (camera/single_usb_stereo_camera.py:311-359), in three parts:
// front = rectify + gray + BT operands + both matchers' cost volumes and horizontal paths;
// middle = the previous-row paths (depth_rest: direction-split on the frame's lane; the grouped frame pipeline:
//          one cluster-fused launch per pass over a lane set's volumes);
// back  = WTA / LR check / median / speckles of both matchers + WLS + depth.
struct DepthRuns {
    SgbmRun left, right;
    bool has_right = false;
    bool vwave = false;  // the grouped pipeline aggregates this frame's volumes with the wavefront kernel
};
int depth_front(Lane& L, const l3d_depth_config& cfg, const RectMap* maps, const uint8_t* lsrc, const uint8_t* rsrc,
                int W, int H, long stride, uint8_t* rectL, DepthRuns& dr);
int depth_back(Lane& L, const l3d_depth_config& cfg, DepthRuns& dr, int W, int H, float* depth, int16_t* disp_f);
// middle + back of one frame start to finish on its lane
int depth_rest(Lane& L, const l3d_depth_config& cfg, DepthRuns& dr, int W, int H, float* depth, int16_t* disp_f);

}  // namespace l3d
