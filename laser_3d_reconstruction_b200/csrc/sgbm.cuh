// sgbm.cuh -- types shared by the StereoSGBM translation units (sgbm_cost.cu, sgbm.cu) and the C ABI's (api.cu,
// pipeline.cu, through api.cuh).
// Internal to libl3d.so.
#pragma once
#include "common.cuh"

namespace l3d {

constexpr int MAXSEG = 4;

// geometry of one matcher run (cv2.StereoSGBM parameter rules, SURVEY A3/A4)
struct Geom {
    int W, H, minD, D, maxD, minX1, maxX1, width1, bs, SW2, P1, P2, uniq, d12, ftzero, mode;
    int DPL, NP, nact;
    int HV, nseg;
    int seg_vr0[MAXSEG], seg_y0[MAXSEG], seg_rows[MAXSEG], seg_emit[MAXSEG];
    int seg_shift[MAXSEG];  // SGBM_3WAY on images of a few rows: output row = computed row - shift (make_geom)
};
int make_geom(const l3d_sgbm_params& p, int W, int H, Geom& g, std::string* err);
// columns of the cost volume: maxX1 - minX1 of make_geom (<= 0: no column has a full disparity range)
inline int sgbm_width1(const l3d_sgbm_params& p, int W) {
    return (W + std::min(p.minDisparity, 0)) - std::max(p.minDisparity + p.numDisparities, 0);
}

// One matcher run = front (BT operands, cost volume, both horizontal paths)
//                 + middle (the previous-row paths: cluster-fused or direction-split)
//                 + back (WTA if not fused, LR check, median, speckles).
struct SgbmRun {
    l3d_sgbm_params p;
    Geom g;
    int W = 0, H = 0;
    int16_t* C = nullptr;
    int16_t* S = nullptr;
    int16_t* raw = nullptr;
    unsigned* d2 = nullptr;
    uint2* wrec = nullptr;   // per-pixel winner records of the wavefront kernel's last pass (behind d2 in the same scratch slot)
    bool wta_done = false;
    bool no_hpair = false;  // the horizontal paths are aggregated by the wavefront kernel (sgbm_vwave.cu), not in the front
};

// ---- sgbm_cost.cu
// BT operand planes of one view (two planes of W*H uint4, see sgbm_prefilter_kernel)
int sgbm_prefilter(Lane& L, const uint8_t* img, int W, int H, int ftzero, uint4* desc);
// cost volume of one run: C = P2 + box sum of the BT pixel cost (descL / descR = operands of the run's own left / right view)
int sgbm_cost_single(Lane& L, const Geom& g, const uint4* descL, const uint4* descR, int16_t* C);
// Both matchers' cost volumes of one frame from ONE pixel-cost pass (gl = left matcher, minD = 0; gr = right matcher,
// minD = -(D-1), views swapped): false when the pair of geometries is not covered (caller runs two single passes)
bool sgbm_cost_dual_ok(const Geom& gl, const Geom& gr);
int sgbm_cost_dual(Lane& L, const Geom& gl, const Geom& gr, const uint4* descLeftView, const uint4* descRightView,
                   int16_t* Cl, int16_t* Cr);

// ---- sgbm.cu
int sgbm_front(Lane& L, const l3d_sgbm_params& p, const uint8_t* left, const uint8_t* right, int W, int H, int set,
               uint4* dL, uint4* dR, bool make_desc, SgbmRun& r);
// left + right matcher of one frame (views swapped for the right one) with the shared pixel-cost pass when covered
int sgbm_front_pair(Lane& L, const l3d_sgbm_params& pl, const l3d_sgbm_params& pr, const uint8_t* left,
                    const uint8_t* right, int W, int H, uint4* dL, uint4* dR, SgbmRun& rl, SgbmRun& rr);
bool sgbm_vgroup_ok(const SgbmRun& r);
int sgbm_middle_split(Lane& L, SgbmRun& r, bool keep_S);
int sgbm_middle_vgroup(Lane& L, SgbmRun* const* runs, int nruns, bool keep_S);
// all eight paths of MODE_HH in two wavefront passes (runs fronted with no_hpair)
bool sgbm_vwave_ok(int width1, int H, int D, int mode);
int sgbm_middle_vwave(Lane& L, SgbmRun* const* runs, int nruns);
int sgbm_back(Lane& L, SgbmRun& r, int16_t* disp, SgbmDebug* dbg);

}  // namespace l3d
