// pipeline.cu -- the frame pipeline of include/l3d.h (l3d_pipeline_*): nframes independent frames over `lanes` streams.
#include <chrono>
#include <stdexcept>

#include "api.cuh"

using namespace l3d;

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
    // The schedule, fixed when the pipeline is created (pipe_plan).
    struct Plan {
        bool grouped = false;  // lane sets with cluster-fused aggregation (else each frame start to finish on its lane)
        int gsz = 1;           // frames per lane set
        bool vwave = false;    // grouped middles run the wavefront kernel (sgbm_vwave.cu), else sgbm_vgroup
    } plan;
    // grouped mode: the frames of a lane set run their SGBM fronts on their lanes, ONE cluster-fused
    // aggregation launch per pass over all their volumes on the set's middle stream, then their backs
    static constexpr int MAXSETS = 8;
    Lane mid[MAXSETS];
    cudaEvent_t ev_mid[MAXSETS] = {};
    std::vector<cudaEvent_t> lane_front;
    std::vector<DepthRuns> runs;  // per lane
    bool timing = false;
    // Steady-state replay: a step with the same buffers and frame count as the previous one is captured once
    // (all lane / aggregation / back streams fork from and join `main`) and replayed as a CUDA graph -- the
    // 34 launches per frame otherwise make small configurations (320x360) host-launch-bound.
    struct GraphKey {
        const void *left, *right, *depth_h, *xyz_h; int nframes; bool host_in; int split;
        bool operator==(const GraphKey& o) const {
            return left == o.left && right == o.right && depth_h == o.depth_h && xyz_h == o.xyz_h && nframes == o.nframes &&
                   host_in == o.host_in && split == o.split;
        }
    };
    struct GraphEntry { GraphKey key; int seen = 0; bool launch_bound = false; cudaGraphExec_t exec = nullptr; long long launches = 0; };
    std::vector<GraphEntry> graphs;
    bool graphs_ok = true;          // cleared when a capture fails: the pipeline then stays on direct launches
    long long graph_launches = 0;   // kernel launches performed by graph replays
    long long graph_replays = 0;
    cudaEvent_t ev_fork = nullptr;
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

// Where a step reads its frames.  Separate eyes (split < 0): two packed arrays of W x H x 3 views.  Captures (split 0 / 1,
// include/l3d.h): one array of stereo captures; both views of a frame are strided row sets of its capture, read in place
// by the rectification kernels -- no de-interleaving pass.
struct PipeSrc {
    const uint8_t *left, *right;  // frame 0's views
    size_t step;                  // bytes from a frame's view to the next frame's: W*H*3 for eyes, 2*W*H*3 for captures
    long stride;                  // row stride of a view
    int split;                    // -1 separate eyes, 0 side by side, 1 top / bottom
    bool host;                    // host memory: staged per frame into the lane's scratch
};
static PipeSrc pipe_src_eyes(const l3d_pipeline* p, const uint8_t* left, const uint8_t* right, bool host) {
    const size_t W = p->cfg.W, H = p->cfg.H;
    return PipeSrc{left, right, W * H * 3, 3L * (long)W, -1, host};
}
static PipeSrc pipe_src_captures(const l3d_pipeline* p, const uint8_t* frames, int split, bool host) {
    const size_t W = p->cfg.W, H = p->cfg.H;
    return PipeSrc{frames, frames + (split == 0 ? W * 3 : W * H * 3), 2 * W * H * 3, (split == 0 ? 6L : 3L) * (long)W,
                   split, host};
}
// frame f's two views as device pointers; host frames go up on the lane's stream first: separate eyes as two copies,
// a capture as ONE copy of both views
static int pipe_views(const PipeSrc& s, Lane& L, int f, const uint8_t*& l, const uint8_t*& r) {
    l = s.left + s.step * f;
    r = s.right + s.step * f;
    if (!s.host) return L3D_OK;
    if (s.split < 0) {
        uint8_t* sl = L.get<uint8_t>(S_SRC_L, s.step);
        uint8_t* sr = L.get<uint8_t>(S_SRC_R, s.step);
        L3D_CHECK(L, cudaMemcpyAsync(sl, l, s.step, cudaMemcpyHostToDevice, L.stream));
        L3D_CHECK(L, cudaMemcpyAsync(sr, r, s.step, cudaMemcpyHostToDevice, L.stream));
        l = sl; r = sr;
    } else {
        // a slot of its own: growing S_SRC_L would free the buffer a graph captured for separate eyes reads
        uint8_t* st = L.get<uint8_t>(S_SRC_CAP, s.step);
        L3D_CHECK(L, cudaMemcpyAsync(st, l, s.step, cudaMemcpyHostToDevice, L.stream));
        r = st + (r - l);
        l = st;
    }
    return L3D_OK;
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
    // PLANE reads no image, DEPTH the depth plane (metres), the DISPARITY kinds the int16 x16 disparity the frame
    // returns (WLS-filtered when depth.use_wls): written by the same stream, ahead of this launch, in every mode
    const float* depth = (c.recon.kind == L3D_RECON_PLANE) ? nullptr : o.depth;
    const int16_t* disp = o.disp;
    L.t_begin("recon");
    if (c.recon.kind == L3D_RECON_DISPARITY || c.recon.kind == L3D_RECON_DISPARITY_MEDIAN)
        RC(dev_recon(L, c.recon, xy64, xy32, o.n_xy, c.max_points, disp, W, H, o.xyz, o.n_xyz));
    else
        RC(dev_recon(L, c.recon, xy64, xy32, o.n_xy, c.max_points, depth, W, H, o.xyz, o.n_xyz));
    L.t_end("recon");
    return L3D_OK;
}

// the last work of frame f in both schedules, on L.stream after its depth: the laser points, their counts into the
// pinned count array, and the depth plane and 3D points into the caller's host arrays when given
static int pipe_frame_tail(l3d_pipeline* p, Lane& L, int f, float* depth_h, double* xyz_h) {
    const size_t n = (size_t)p->cfg.W * p->cfg.H, cap = p->cfg.max_points;
    FrameOut& o = p->outs[f];
    RC(pipe_extract(p, L, o));
    L3D_CHECK(L, cudaMemcpyAsync(p->counts_host + 2 * f, o.n_xy, sizeof(int), cudaMemcpyDeviceToHost, L.stream));
    L3D_CHECK(L, cudaMemcpyAsync(p->counts_host + 2 * f + 1, o.n_xyz, sizeof(int), cudaMemcpyDeviceToHost, L.stream));
    if (depth_h) L3D_CHECK(L, cudaMemcpyAsync(depth_h + n * f, o.depth, n * 4, cudaMemcpyDeviceToHost, L.stream));
    if (xyz_h) L3D_CHECK(L, cudaMemcpyAsync(xyz_h + cap * 3 * f, o.xyz, cap * 24, cudaMemcpyDeviceToHost, L.stream));
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

// The schedule.  Grouped mode: one aggregation launch should carry close to (but not more than) one wave of clusters --
// 15 clusters of 8 CTAs (14 of 9) are resident on a B200 (cudaOccupancyMaxActiveClusters) -- so a lane set is
// 7 frames with WLS (14 volumes) or 15 without; up to 4 sets alternate to overlap fronts/backs with
// another set's aggregation.  3WAY / HH4, fewer lanes than 8 volumes and geometries the cluster kernels do not
// cover run each frame start to finish on its lane (direction-split).
constexpr int VG_WAVE = 15;
static l3d_pipeline::Plan pipe_plan(const l3d_pipeline_config& c) {
    const l3d_sgbm_params& q = c.depth.left;
    const int jobs_per_frame = c.depth.use_wls ? 2 : 1, width1 = sgbm_width1(q, c.W);
    l3d_pipeline::Plan pl;
    pl.gsz = std::min(c.lanes, std::max(1, VG_WAVE / jobs_per_frame));
    pl.grouped = pl.gsz * jobs_per_frame >= 8 && q.mode < 2 && width1 > 0 && vgroup_supported(width1, c.H, q.numDisparities);
    pl.vwave = pl.grouped && sgbm_vwave_ok(width1, c.H, q.numDisparities, q.mode);
    return pl;
}

// the first m 2-D points of a frame into a float or double array: the Simple extractor stores them as double, Steger
// as float
template <typename T>
static cudaError_t pipe_copy_xy(const l3d_pipeline* p, const FrameOut& o, int m, T* xy) {
    const bool f64 = p->cfg.extractor == 4;
    const void* src = f64 ? (const void*)o.xy64 : (const void*)o.xy;
    const size_t n = (size_t)2 * m;
    if (f64 == std::is_same<T, double>::value) return cudaMemcpy(xy, src, n * sizeof(T), cudaMemcpyDeviceToHost);
    using Stored = typename std::conditional<std::is_same<T, double>::value, float, double>::type;
    std::vector<Stored> t(n);
    const cudaError_t e = cudaMemcpy(t.data(), src, n * sizeof(Stored), cudaMemcpyDeviceToHost);
    for (size_t i = 0; e == cudaSuccess && i < n; i++) xy[i] = (T)t[i];
    return e;
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
    if (cfg->recon.kind == L3D_RECON_DISPARITY_MEDIAN) NEED(ctx, recon_window_ok(cfg->recon.window), "median window must be odd, <= 9");
    CK(ctx, cudaSetDevice(ctx->device));
    l3d_pipeline* p = new l3d_pipeline();
    p->ctx = ctx; p->cfg = *cfg;
    p->plan = pipe_plan(*cfg);
    p->lanes.resize(cfg->lanes);
    // Stream priorities.  The cluster-fused aggregation needs 8 completely free SMs of one GPC per volume, so its
    // launches go first whenever they are ready (any resident CTA of another kernel blocks a cluster CTA: it takes
    // the whole register file); the short back-half kernels come next, the wide front kernels fill the rest.
    int prio_lo = 0, prio_hi = 0;
    CK(ctx, cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    const int prio[3] = {prio_hi, prio_lo, std::max(prio_hi, prio_lo - 2)};  // aggregation, front, back
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

static int pipe_run_grouped(l3d_pipeline* p, const PipeSrc& src, int nframes, float* depth_h, double* xyz_h) {
    l3d_ctx* ctx = p->ctx;
    const l3d_pipeline_config& c = p->cfg;
    const int W = c.W, H = c.H;
    const int nl = (int)p->lanes.size();
    const int gsz = p->plan.gsz;
    const int nsets = p->timing ? 1 : std::max(1, std::min(l3d_pipeline::MAXSETS, nl / gsz));  // lane sets alternate
    const int nchunks = (nframes + gsz - 1) / gsz;
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
            if (p->timing && i > 0) CK(ctx, cudaStreamWaitEvent(L.stream, p->lane_front[li - 1], 0));  // kernels alone
            const uint8_t *l, *r;
            RC(pipe_views(src, L, f, l, r));
            DepthRuns& dr = p->runs[li];
            dr.vwave = p->plan.vwave;
            RC(depth_front(L, c.depth, p->maps, l, r, W, H, src.stride, p->outs[f].rect, dr));
            CK(ctx, cudaEventRecord(p->lane_front[li], L.stream));
            CK(ctx, cudaStreamWaitEvent(M.stream, p->lane_front[li], 0));
            list.push_back(&dr.left);
            if (dr.has_right) list.push_back(&dr.right);
        }
        if (p->plan.vwave) RC(sgbm_middle_vwave(M, list.data(), (int)list.size()));
        else RC(sgbm_middle_vgroup(M, list.data(), (int)list.size(), false));
        CK(ctx, cudaEventRecord(p->ev_mid[set], M.stream));
        for (int i = 0; i < ng; i++) {
            const int li = set * gsz + i, f = f0 + i;
            Lane& L = p->lanes[li];
            // the back half runs on the lane's second stream (own priority); the lane's main stream rejoins below
            cudaStream_t front_stream = L.stream;
            if (!p->timing) {
                CK(ctx, cudaStreamWaitEvent(L.back_stream, p->lane_front[li], 0));
                L.stream = L.back_stream;
            }
            struct Restore { Lane& l; cudaStream_t s; ~Restore() { l.stream = s; } } restore{L, front_stream};
            CK(ctx, cudaStreamWaitEvent(L.stream, p->ev_mid[set], 0));
            if (p->timing && i > 0) CK(ctx, cudaStreamWaitEvent(L.stream, p->lane_done[li - 1], 0));
            RC(depth_back(L, c.depth, p->runs[li], W, H, p->outs[f].depth, p->outs[f].disp));
            RC(pipe_frame_tail(p, L, f, depth_h, xyz_h));
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
static int pipe_enqueue(l3d_pipeline* p, const PipeSrc& src, int nframes, float* depth_h, double* xyz_h) {
    l3d_ctx* ctx = p->ctx;
    const l3d_pipeline_config& c = p->cfg;
    const int nl = (int)p->lanes.size();
    CK(ctx, cudaEventRecord(p->ev_fork, p->main));
    for (auto& L : p->lanes) CK(ctx, cudaStreamWaitEvent(L.stream, p->ev_fork, 0));
    if (p->plan.grouped) RC(pipe_run_grouped(p, src, nframes, depth_h, xyz_h));
    else for (int f = 0; f < nframes; f++) {  // each frame start to finish on its lane
        Lane& L = p->lanes[f % nl];
        FrameOut& o = p->outs[f];
        const uint8_t *l, *r;
        RC(pipe_views(src, L, f, l, r));
        DepthRuns dr;
        dr.vwave = p->plan.vwave;
        RC(depth_front(L, c.depth, p->maps, l, r, c.W, c.H, src.stride, o.rect, dr));
        RC(depth_rest(L, c.depth, dr, c.W, c.H, o.depth, o.disp));
        RC(pipe_frame_tail(p, L, f, depth_h, xyz_h));
    }
    for (int i = 0; i < nl; i++) {
        CK(ctx, cudaEventRecord(p->lane_done[i], p->lanes[i].stream));
        CK(ctx, cudaStreamWaitEvent(p->main, p->lane_done[i], 0));
    }
    return L3D_OK;
}

// launches enqueued on the lanes and aggregation streams (directly or into a captured graph)
static long long pipe_launches_now(const l3d_pipeline* p) {
    long long s = 0;
    for (auto& L : p->lanes) s += L.launches;
    for (int i = 0; i < l3d_pipeline::MAXSETS; i++) s += p->mid[i].launches;
    return s;
}

static int pipe_run(l3d_pipeline* p, const PipeSrc& src, int nframes, float* depth_h, double* xyz_h, int* counts) {
    l3d_ctx* ctx = p->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    RC(pipe_prepare(p, nframes));
    for (auto& L : p->lanes) L.t_reset();
    auto t_enq0 = std::chrono::steady_clock::now();
    // ---- CUDA-graph replay of a repeated step (same buffers and input form, same frame count); the first occurrence
    // runs with direct launches (it also grows the scratch buffers), the second decides whether the step is
    // launch-bound, the third is captured, later ones are replayed
    static const bool graphs_off = (getenv("L3D_NO_GRAPH") && atoi(getenv("L3D_NO_GRAPH")) > 0) || getenv("L3D_DEBUG_SKIP");
    l3d_pipeline::GraphEntry* ge = nullptr;
    if (!graphs_off && p->graphs_ok && !p->timing) {
        const l3d_pipeline::GraphKey key{src.left, src.right, depth_h, xyz_h, nframes, src.host, src.split};
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
                rc = pipe_enqueue(p, src, nframes, depth_h, xyz_h);
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
        RC(pipe_enqueue(p, src, nframes, depth_h, xyz_h));
    }
    CK(ctx, cudaEventRecord(p->ev1, p->main));
    const double enq_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_enq0).count();
    CK(ctx, cudaEventSynchronize(p->ev1));
    CK(ctx, cudaEventElapsedTime(&p->last_ms, p->ev0, p->ev1));
    // a step whose direct enqueue takes a large part of its GPU time is launch-bound: replay it as a graph from now on
    // (at config 3 the enqueue is 12 % of the step and direct launches with stream priorities are 2 % faster)
    // (judged on the second occurrence: the first one also allocates the scratch buffers)
    if (ge && !replayed && ge->seen == 2) ge->launch_bound = enq_ms > 0.4 * (double)p->last_ms;
    p->last_frames = nframes;
    if (counts) for (int f = 0; f < nframes; f++) counts[f] = p->counts_host[2 * f + 1];
    return check_flags(ctx, p->flags);
}

int l3d_pipeline_run_dev(l3d_pipeline* p, const uint8_t* left_dev, const uint8_t* right_dev, int nframes, int* counts) {
    if (!p) return L3D_ERR_ARG;
    l3d_ctx* ctx = p->ctx;
    API_BEGIN(ctx)
    NEED(ctx, left_dev && right_dev && nframes > 0, "pipeline_run_dev arguments");
    return pipe_run(p, pipe_src_eyes(p, left_dev, right_dev, false), nframes, nullptr, nullptr, counts);
    API_END(ctx)
}

int l3d_pipeline_run_host(l3d_pipeline* p, const uint8_t* left, const uint8_t* right, int nframes, float* depth,
                          double* xyz, int* counts) {
    if (!p) return L3D_ERR_ARG;
    l3d_ctx* ctx = p->ctx;
    API_BEGIN(ctx)
    NEED(ctx, left && right && nframes > 0, "pipeline_run_host arguments");
    return pipe_run(p, pipe_src_eyes(p, left, right, true), nframes, depth, xyz, counts);
    API_END(ctx)
}

int l3d_pipeline_run_captures_dev(l3d_pipeline* p, const uint8_t* frames_dev, int nframes, int split, int* counts) {
    if (!p) return L3D_ERR_ARG;
    l3d_ctx* ctx = p->ctx;
    API_BEGIN(ctx)
    NEED(ctx, frames_dev && nframes > 0 && (split == 0 || split == 1), "pipeline_run_captures_dev arguments");
    return pipe_run(p, pipe_src_captures(p, frames_dev, split, false), nframes, nullptr, nullptr, counts);
    API_END(ctx)
}

int l3d_pipeline_run_captures_host(l3d_pipeline* p, const uint8_t* frames, int nframes, int split, float* depth,
                                   double* xyz, int* counts) {
    if (!p) return L3D_ERR_ARG;
    l3d_ctx* ctx = p->ctx;
    API_BEGIN(ctx)
    NEED(ctx, frames && nframes > 0 && (split == 0 || split == 1), "pipeline_run_captures_host arguments");
    return pipe_run(p, pipe_src_captures(p, frames, split, true), nframes, depth, xyz, counts);
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
    if (xy && m > 0) CK(ctx, pipe_copy_xy(p, o, m, xy));
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
    if (xy && m > 0) CK(ctx, pipe_copy_xy(p, o, m, xy));
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

long long l3d_pipeline_launch_count(l3d_pipeline* p) { return p ? pipe_launches_now(p) + p->graph_launches : 0; }

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
