// sgbm_vwave.cu -- host side of the wavefront aggregation (kernel: sgbm_vwave.cuh) and its D <= 128 instantiations
#include <map>
#include <mutex>

#include "sgbm_vwave.cuh"

namespace l3d {

// How many clusters of `cluster` CTAs of the (last-pass) kernel can be resident at once on the current device
// (cudaOccupancyMaxActiveClusters; cached per device and shape).  B200s differ in how their 148 SMs are spread over the
// GPCs, and a cluster lives inside one GPC: a 20- or 18-SM GPC holds two 9-CTA clusters, a 16-SM GPC only one.
template <int NP, int CPW>
static int vwave_resident_query(int cluster, size_t smem) {
    auto kern = sgbm_vwave_kernel<NP, CPW, true, true, 16>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
        cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(cluster, VW_MAXJOBS);
    cfg.blockDim = dim3(16 * 32);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
static int vwave_resident_clusters(int D, int cpw, int cluster) {
    static std::mutex mu;
    static std::map<long long, int> cache;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return 0; }
    const long long key = (((long long)dev * 512 + D) * 64 + cpw) * 64 + cluster;
    std::lock_guard<std::mutex> g(mu);
    auto it = cache.find(key);
    if (it != cache.end()) return it->second;
    const size_t smem = vwave_smem_bytes(D, cpw, true);
    int n = 0;
#define VW_Q(NPV, CPWV) if (D == 64 * NPV && cpw == CPWV) n = vwave_resident_query<NPV, CPWV>(cluster, smem);
#define VW_QN(NPV) VW_Q(NPV, 2) VW_Q(NPV, 3) VW_Q(NPV, 4) VW_Q(NPV, 5) VW_Q(NPV, 6) VW_Q(NPV, 7) VW_Q(NPV, 8) VW_Q(NPV, 9)
    VW_QN(1) VW_QN(2)
#undef VW_QN
#undef VW_Q
    cache[key] = n;
    return n;
}

// geometry -> (CTAs per cluster, columns per warp).  D <= 128: 16 warps per CTA, 2..9 columns per warp, a 9-CTA cluster
// where it fits exactly (below), else the smallest of an 8- or a 16-CTA cluster that covers width1; D = 256: 8 warps per
// CTA, 16-CTA cluster, 10..13 columns per warp (narrower volumes stay on the other kernels: the instantiations are
// expensive)
static bool vwave_shape(int width1, int D, int& cluster, int& cpw) {
    if (D == 256) {
        const int c = cdiv(width1, 16 * vwave_warps(D));
        if (c < 10 || c > VW_MAXCPW256 || vwave_smem_bytes(D, c, true) > 227 * 1024) return false;
        cluster = 16; cpw = c;
        return true;
    }
    if (!(D == 64 || D == 128)) return false;
    // Nine CTAs where they cover the volume exactly with fewer columns per warp than eight would need (config 3: 1152 =
    // 9 x 16 x 8 instead of 8 x 16 x 9).  Two 9-CTA clusters fit a 20-SM GPC like two 8-CTA ones, so the 14 volumes of a
    // lane set are still one wave, on 126 SMs instead of 112: 0.141 + 0.181 -> 0.126 + 0.161 ms per run alone; the frame
    // pipeline, whose other streams were using the 36 free SMs, is unchanged (1124 vs 1119 frames/s).
    if (width1 % (9 * vwave_warps(D)) == 0) {
        const int c = width1 / (9 * vwave_warps(D));
        // ... provided this GPU keeps a lane set's 14 volumes resident as 9-CTA clusters too (one wave per launch)
        if (c >= 2 && c < cdiv(width1, 8 * vwave_warps(D)) && c <= VW_MAXCPW && vwave_smem_bytes(D, c, true) <= 227 * 1024 &&
            vwave_resident_clusters(D, c, 9) >= 14) {
            cluster = 9; cpw = c;
            return true;
        }
    }
    for (int cl = 8; cl <= 16; cl *= 2) {
        const int c = cdiv(width1, cl * vwave_warps(D));
        if (c <= VW_MAXCPW && c >= 2 && vwave_smem_bytes(D, c, true) <= 227 * 1024) { cluster = cl; cpw = c; return true; }
    }
    return false;
}

bool vwave_supported(int width1, int H, int D) {
    int cl, cpw;
    return width1 >= 1 && H >= 1 && vwave_shape(width1, D, cl, cpw);
}

// Does the wavefront kernel beat horizontal pair + cluster-fused passes on this geometry?  Measured in the frame pipeline
// (frames/s with / without, MODE_HH + WLS, 28 lanes; gpurun_out/geoms.log): 1280x720 D=128 +18 %, 1280x360 D=128 +14 %,
// 960x540 D=128 (7 columns per warp) +7.5 %, 640x480 D=128 (4) +5.5 %, 512x512 D=128 (3) -4 %; D=64: 800x600 -1 %,
// 640x480 -1.5 %, 320x360 (2 columns per warp) -9 %.  The fill and drain of the wavefront (one horizontal chain + hand-off
// per strip) do not shrink with the strips, and at D=64 the bytes the other kernels move twice are half as many.
bool vwave_pays(int width1, int H, int D) {
    int cl, cpw;
    if (!(width1 >= 1 && H >= 1 && vwave_shape(width1, D, cl, cpw))) return false;
    if (D == 256) return true;   // config 4 (13 columns per warp): see DESIGN.md for the measurement
    return D == 128 && cpw >= 4;
}

// The per-pixel tail of the winner-takes-all for all volumes of a last-pass launch: disp2 vote (order-independent atomicMax
// key, sgbm.cu), OpenCV's sub-pixel step with its truncating division, raw disparity.  One thread per pixel over the dense
// records the last pass left.
struct VWaveFinishArgs {
    const uint2* rec[VW_MAXJOBS];
    int16_t* raw[VW_MAXJOBS];
    unsigned* d2[VW_MAXJOBS];
    int minD[VW_MAXJOBS], minX1[VW_MAXJOBS];
    int width1, H, D, W;
};
__global__ void __launch_bounds__(256) vw_finish_kernel(const VWaveFinishArgs a) {
    const int job = blockIdx.y;
    const int n = a.width1 * a.H;
    const int minD = a.minD[job], minX1 = a.minX1[job];
    const uint2* __restrict__ recs = a.rec[job];
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) {
        const uint2 rec = recs[i];
        if (rec.x == 0xffffffffu) continue;
        const int y = i / a.width1, x = i - y * a.width1;
        const int minS = (int)(rec.x >> 8), d = (int)(rec.x & 255u);
        const int x2 = x + minX1 - d - minD;
        if (x2 >= 0 && x2 < a.W + 2)
            atomicMax(a.d2[job] + (size_t)y * (a.W + 2) + x2, ((unsigned)(0x7fff - minS) << 16) | (unsigned)x);
        int dd = d * 16;
        if (0 < d && d < a.D - 1) {
            const int sm = (int)(rec.y & 0xffffu), sp = (int)(rec.y >> 16);
            const int denom2 = max(sm + sp - 2 * minS, 1);
            dd += ((sm - sp) * 16 + denom2) / (denom2 * 2);
        }
        a.raw[job][(size_t)y * a.W + x + minX1] = (int16_t)(dd + minD * 16);
    }
}

// Aggregate four paths of pass `dir` for `njobs` volumes at once; wta != nullptr: last pass (S is read, accumulated,
// reduced by the winner-takes-all and NOT written back), else first pass (S is written, not read).
int dev_sgbm_vwave(Lane& L, const int16_t* const* C, int16_t* const* S, int njobs, int width1, int H, int D, int P1,
                   int P2, int dir, const VGroupWta* wta) {
    int cl = 0, cpw = 0;
    L3D_ARG(L, H >= 1 && vwave_shape(width1, D, cl, cpw), "vwave geometry");
    L3D_ARG(L, (dir > 0) == (wta == nullptr), "vwave: pass 1 runs top-down without the WTA, pass 2 bottom-up with it");
    for (int j0 = 0; j0 < njobs; j0 += VW_MAXJOBS) {
        VWaveArgs a;
        const int nj = std::min(VW_MAXJOBS, njobs - j0);
        for (int j = 0; j < nj; j++) {
            a.C[j] = C[j0 + j]; a.S[j] = S[j0 + j];
            a.rec[j] = nullptr; a.uniq[j] = 0;
            if (wta) {
                L3D_ARG(L, wta[j0 + j].rec != nullptr, "vwave: the last pass needs a record buffer");
                a.rec[j] = wta[j0 + j].rec; a.uniq[j] = wta[j0 + j].uniq;
            }
        }
        a.W = wta ? wta[0].W : 0; a.zero = 0;
        a.width1 = width1; a.H = H; a.D = D; a.P1 = P1; a.P2 = P2; a.dir = dir; a.cluster = cl;
        const bool last = wta != nullptr, full = width1 % cpw == 0;
        const size_t smem = vwave_smem_bytes(D, cpw, last);
        int rc = L3D_ERR_UNSUPPORTED;
        if (D == 256) rc = vwave_launch_256(L, a, cpw, nj, last, full, smem);
#define VW_CASE(NPV, CPWV) else if (D == 64 * NPV && cpw == CPWV) rc = vwave_launch_shape<NPV, CPWV, 16>(L, a, nj, last, full, smem);
#define VW_NP(NPV) VW_CASE(NPV, 2) VW_CASE(NPV, 3) VW_CASE(NPV, 4) VW_CASE(NPV, 5) VW_CASE(NPV, 6) VW_CASE(NPV, 7) \
                   VW_CASE(NPV, 8) VW_CASE(NPV, 9)
        VW_NP(1) VW_NP(2)
#undef VW_NP
#undef VW_CASE
        if (rc != L3D_OK) return rc;
        if (wta) {
            VWaveFinishArgs f;
            for (int j = 0; j < nj; j++) {
                f.rec[j] = wta[j0 + j].rec; f.raw[j] = wta[j0 + j].raw; f.d2[j] = wta[j0 + j].d2;
                f.minD[j] = wta[j0 + j].minD; f.minX1[j] = wta[j0 + j].minX1;
            }
            f.width1 = width1; f.H = H; f.D = D; f.W = a.W;
            L3D_LAUNCH(L, vw_finish_kernel, dim3(std::min(cdiv(width1 * H, 256 * 4), 1024), nj), 256, 0, f);
        }
    }
    return L3D_OK;
}

}  // namespace l3d
