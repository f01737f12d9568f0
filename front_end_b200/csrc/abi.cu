// C-ABI layer: context, device memory, H2D/D2H staging, stage sequencing and per-stage timing.
// Entry points are documented in include/fe_abi.h with the reference interface each one replaces.
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "fe_internal.cuh"

using namespace fe;

namespace {

enum Stage { ST_H2D = 0, ST_FAST, ST_SELECT, ST_ORIENT, ST_BLUR, ST_BRIEF, ST_SURF, ST_KNN, ST_MATCH, ST_L2, ST_L2TC, ST_L2AUX, ST_FINALIZE, ST_D2H, ST_COUNT };
const char *kStageNames[ST_COUNT] = {"h2d", "fast", "select", "orient_pack", "gauss7", "rbrief", "surf_describe",
                                     "hamming_knn2", "hamming_cross", "l2_match_fp32", "l2_tensor", "l2_prep_rerank", "finalize", "d2h"};

thread_local std::string g_create_error;

}  // namespace

struct fe_ctx {
    fe_config cfg{};
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    Buffers b;
    unsigned allocated = 0;   // BufGroup bits of the allocated buffer groups
    Geom g{};                 // geometry of the batch currently resident on the device
    Geom gmax{};              // capacity geometry (fe_config.max_*): what the buffers are sized for
    uint32_t *h_counts = nullptr;   // pinned: [3 * max_images]
    // chunked pipeline (fe_pipeline_batch): copy-in, two compute lanes, copy-out
    cudaStream_t s_in = nullptr, s_out = nullptr, s_cmp[2] = {nullptr, nullptr};
    // side streams of the pruned cross-check (the multi-index join runs beside the verification scans): one per compute stream
    // (ctx stream, the two pipeline lanes), each with its fork / join events
    cudaStream_t s_aux[3] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_fork[3] = {nullptr, nullptr, nullptr}, ev_join[3] = {nullptr, nullptr, nullptr};
    std::vector<cudaEvent_t> ev_in, ev_done;
    cudaEvent_t ev_sync = nullptr;
    int *h_tc_error = nullptr;      // pinned mirror of Buffers::tc_error (tcgen05 mbarrier timeout)
    int nlevels = 1;                  // ORB pyramid (fe_set_orb_pyramid)
    double scale_factor = 1.2000000476837158;   // (double)1.2f, as cv::ORB stores it
    int wta_k = 2;                    // ORB WTA_K (fe_set_orb_wta_k): 3 / 4 -> two-bit symbols, NORM_HAMMING2
    int score_type = 1;               // cv::ORB scoreType (fe_set_orb_score_type): 0 = HARRIS_SCORE, 1 = FAST_SCORE
    int patch_size = 31;              // ORB patchSize (fe_set_orb_patch_size); != 31 selects the generated pattern
    int chunk_pairs = 0;              // pairs per chunk of the overlapped pipeline (fe_set_chunk_pairs); 0 = default
    int batch_desc = FE_DESC_ORB256;  // what the batched pipeline describes with (fe_set_batch_descriptor)
    bool hessian = false;             // the batched pipeline detects with SURF's Fast-Hessian detector (fe_set_batch_detector)
    fe_surf_params surf{};            // its parameters
    int wu_frames = 0, wu_prev_n = 0;  // fe_window_update: frames in the window, landmarks of the previous frame
    bool wu_prev_sorted = true;
    int wu_dim = 0;                    // rows of the frames in the window: 0 = binary, 64 / 128 = SURF floats
    int brief_bytes[3] = {0, 0, 0};   // fe_set_brief_pattern: table present for BRIEF-16 / 32 / 64 (Buffers::brief_tab)
    int brief_orient[3] = {0, 0, 0};
    // fe_set_freak: cv::FREAK's pattern sizes and parameters (the pattern itself is in Buffers::freak_*)
    int freak_sizes[64] = {0};
    int freak_orient = 1, freak_scale_norm = 1, freak_octaves = 4;
    bool cross_prune = true;        // FE_CROSS_PRUNE=0 forces the all-pairs cross-check kernel (A/B testing)
    bool cross_mih = true;          // FE_CROSS_MIH=0: pruned cross-check without the multi-index join (A/B testing)
    int l2_tensor = 1;              // FE_L2_TENSOR: 0 = FP32 kernels only; 1 = exact tensor-core cross-check (l2verify.cu) where it applies;
                                    // 2 = additionally the approximate tcgen05 top-k candidates (l2tc.cu) for the unmasked cases
    int64_t h2d_bytes = 0, d2h_bytes = 0;   // batched paths only (bench.py's e2e accounting)
    std::string err;
    std::atomic<int> pending_threshold{-1}, pending_setpoint{INT32_MIN};
    // profiling
    bool profiling = false;
    struct Pending { int stage; cudaEvent_t a, b; };
    std::vector<Pending> pending;
    std::vector<cudaEvent_t> pool;
    double stage_ms[ST_COUNT] = {0};
    int64_t stage_launches[ST_COUNT] = {0};
    int64_t launches = 0;
    double last_stage_ms[ST_COUNT] = {0};
};

namespace {

#define FE_CUDA(ctx, call)                                                                        \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess) {                                                                  \
            (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e_);                      \
            return FE_ERR_CUDA;                                                                   \
        }                                                                                         \
    } while (0)

int fail(fe_ctx *ctx, int code, const char *msg) {
    if (ctx) ctx->err = msg;
    return code;
}

// Calls f(pointer member, elements per unit at geometry g, scope, group, name) for every entry of FE_BUFFERS.
template <typename F>
void for_each_buffer(Buffers &b, const Geom &g, F &&f) {
#define FE_VISIT(T, name, scope, group, n) f(b.name, (size_t)(n), scope, (unsigned)group, #name);
    FE_BUFFERS(FE_VISIT)
#undef FE_VISIT
}

// Images, or pairs, among the first n_images images: the units per-image and per-pair buffers are laid out in.
size_t units(BufScope s, int n_images) { return s == PER_IMAGE ? (size_t)n_images : (size_t)(n_images + 1) / 2; }

// Allocates every buffer of the groups in `groups` that is not allocated yet, sized at the capacity geometry, and
// zero-fills it on the ctx stream (a non-blocking stream does not order against the legacy default stream, so a plain
// cudaMemset could land after the kernels that follow).  Each allocation carries 64 bytes of slack past its end, which
// the image kernels' vector loads may touch.
int ensure(fe_ctx *c, unsigned groups) {
    groups &= ~c->allocated;
    if (!groups) return FE_OK;
    cudaError_t e = cudaSuccess;
    for_each_buffer(c->b, c->gmax, [&](auto *&p, size_t n, BufScope s, unsigned grp, const char *name) {
        if (e != cudaSuccess || !(grp & groups) || p || n == 0) return;
        const size_t bytes = (s == PER_CTX ? 1 : units(s, c->gmax.n_images)) * n * sizeof(*p) + 64;
        if ((e = cudaMalloc(reinterpret_cast<void **>(&p), bytes)) == cudaSuccess) e = cudaMemsetAsync(p, 0, bytes, c->stream);
        if (e != cudaSuccess) c->err = std::string("allocating ") + name + ": " + cudaGetErrorString(e);
    });
    if (e != cudaSuccess) return FE_ERR_CUDA;
    c->allocated |= groups;
    return FE_OK;
}

// The buffers of images [first, ...) (first even) of the resident geometry g, seen as a batch of their own.
Buffers view_of(const Buffers &b, const Geom &g, int first) {
    Buffers v = b;
    for_each_buffer(v, g, [&](auto *&p, size_t n, BufScope s, unsigned, const char *) {
        if (p && s != PER_CTX) p += units(s, first) * n;
    });
    return v;
}

cudaEvent_t get_event(fe_ctx *c) {
    if (!c->pool.empty()) {
        cudaEvent_t e = c->pool.back();
        c->pool.pop_back();
        return e;
    }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}

struct StageTimer {
    fe_ctx *c;
    int stage;
    cudaStream_t s;
    bool on;
    cudaEvent_t a = nullptr;
    StageTimer(fe_ctx *ctx, int st) : StageTimer(ctx, st, ctx->stream, true) {}
    // timed = false for work issued on the auxiliary streams of the chunked pipeline (kernels of
    // different chunks overlap there, so per-stage event pairs would not measure one kernel)
    StageTimer(fe_ctx *ctx, int st, cudaStream_t stream, bool timed) : c(ctx), stage(st), s(stream), on(timed && ctx->profiling) {
        if (on) {
            a = get_event(c);
            cudaEventRecord(a, s);
        }
    }
    void done(int n_launches) {
        c->launches += n_launches;
        c->stage_launches[stage] += n_launches;
        if (on) {
            cudaEvent_t b = get_event(c);
            cudaEventRecord(b, s);
            c->pending.push_back({stage, a, b});
        }
    }
};

// Fold finished event pairs into the per-stage totals (stream must be synchronised).
void resolve_pending(fe_ctx *c) {
    for (int i = 0; i < ST_COUNT; ++i) c->last_stage_ms[i] = 0;
    for (auto &p : c->pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) {
            c->stage_ms[p.stage] += ms;
            c->last_stage_ms[p.stage] += ms;
        }
        c->pool.push_back(p.a);
        c->pool.push_back(p.b);
    }
    c->pending.clear();
}

Geom geom_of(const fe_config &cfg, int w, int h, int n_images) {
    Geom g{};
    g.w = w; g.h = h; g.pitch = round_up(w, 16);
    g.n_images = n_images;
    set_strip_geometry(g, cfg.nonmax != 0);
    g.kp_cap = cfg.max_keypoints;
    g.img_stride = (size_t)g.pitch * h;
    g.rs_h = cfg.max_height;
    return g;
}

int set_geom(fe_ctx *c, int w, int h, int n_images) {
    if (w < 1 || h < 1 || n_images < 1) return fail(c, FE_ERR_BAD_ARG, "non-positive image geometry");
    if (w > c->cfg.max_width || h > c->cfg.max_height)
        return fail(c, FE_ERR_BAD_ARG, "image larger than fe_config.max_width/max_height");
    if (n_images > c->cfg.max_images)
        return fail(c, FE_ERR_CAPACITY, "batch larger than fe_config.max_images");
    c->g = geom_of(c->cfg, w, h, n_images);
    return FE_OK;
}

void apply_pending_detection(fe_ctx *c) {
    const int t = c->pending_threshold.exchange(-1);
    if (t >= 1) c->cfg.fast_threshold = t;
    const int sp = c->pending_setpoint.exchange(INT32_MIN);
    if (sp != INT32_MIN) c->cfg.n_features = sp;
}

DetectParams detect_params(const fe_ctx *c) {
    DetectParams p;
    p.threshold = c->cfg.fast_threshold;
    p.ps = c->cfg.fast_type;
    p.nonmax = c->cfg.nonmax;
    p.n_features = c->cfg.n_features;
    p.edge = c->cfg.edge_threshold;
    p.patch_size = c->patch_size;
    p.wta_k = c->wta_k;
    return p;
}

// Upload n contiguous host images (row stride `stride`) into device image slots first, first+step, ...
int upload_images(fe_ctx *c, const uint8_t *src, int n, int stride, int first, int step) {
    const Geom &g = c->g;
    if (stride == g.w && g.pitch == g.w) {
        // every image is one contiguous run on both sides: a single strided copy
        FE_CUDA(c, cudaMemcpy2DAsync(c->b.img + (size_t)first * g.img_stride, (size_t)step * g.img_stride,
                                     src, g.img_stride, g.img_stride, n, cudaMemcpyHostToDevice, c->stream));
    } else {
        for (int i = 0; i < n; ++i)
            FE_CUDA(c, cudaMemcpy2DAsync(c->b.img + (size_t)(first + i * step) * g.img_stride, g.pitch,
                                         src + (size_t)i * stride * g.h, stride, g.w, g.h,
                                         cudaMemcpyHostToDevice, c->stream));
    }
    return FE_OK;
}

// HARRIS_SCORE only exists inside cv::ORB's detector (orientation mode with a setpoint)
bool use_harris(const fe_ctx *c) { return c->score_type == 0 && c->cfg.orientation && c->cfg.n_features >= 0; }

// detect (+ optional describe) for the images resident on the device
int run_detect_on(fe_ctx *c, const Geom &g, const Buffers &b, cudaStream_t st, bool describe, bool timed) {
    DetectParams p = detect_params(c);
    const bool harris = use_harris(c);
    const int n_final = p.n_features;
    if (harris && n_final > 0) {
        // "keep more points than necessary", orb.cpp computeKeyPoints: the Harris cut needs all 2N candidates resident
        if (2 * (long long)n_final > g.kp_cap)
            return fail(c, FE_ERR_CAPACITY, "HARRIS_SCORE keeps 2 x n_features FAST corners before the Harris cut: raise fe_config.max_keypoints");
        p.n_features = 2 * n_final;
    }
    { StageTimer t(c, ST_FAST, st, timed); t.done(launch_fast(g, p, b, st)); }
    { StageTimer t(c, ST_SELECT, st, timed); t.done(launch_select(g, p, b, st)); }
    if (harris) { StageTimer t(c, ST_SELECT, st, timed); t.done(launch_harris_select(g, n_final, b, st)); }
    // default ORB geometry: orientation and rBRIEF in one pass over image tiles, after the blur (which needs no keypoints)
    if (describe && c->cfg.orientation && !harris && describe_tile_fits(p)) {
        { StageTimer t(c, ST_BLUR, st, timed); t.done(launch_blur(g, b, st)); }
        { StageTimer t(c, ST_BRIEF, st, timed); t.done(launch_describe_tile(g, p, b, st)); }
        FE_CUDA(c, cudaGetLastError());
        return FE_OK;
    }
    { StageTimer t(c, ST_ORIENT, st, timed); t.done(launch_orient(g, p, b, c->cfg.orientation != 0, st)); }
    if (harris) { StageTimer t(c, ST_ORIENT, st, timed); t.done(launch_harris_store(g, b, st)); }
    if (describe) {
        { StageTimer t(c, ST_BLUR, st, timed); t.done(launch_blur(g, b, st)); }
        { StageTimer t(c, ST_BRIEF, st, timed); t.done(launch_rbrief(g, p, b, b.n_kp, st)); }
    }
    FE_CUDA(c, cudaGetLastError());
    return FE_OK;
}

int cv_round_f(float v) { return (int)lrint((double)v); }

// cv::ORB::detectAndCompute with nlevels > 1 for the images resident at level-0 geometry (pyramid.cu).  Results end up in
// the same arrays the single-level path fills (b.kp, b.desc, b.n_kp, b.kx, b.ky), level-major.
int run_detect_pyramid(fe_ctx *c, bool describe) {
    const Geom g0 = c->g;
    Buffers &b = c->b;
    const int NI = g0.n_images, L = c->nlevels;
    { const int r = ensure(c, GRP_PYRAMID); if (r != FE_OK) return r; }
    FE_CUDA(c, cudaMemsetAsync(b.pyr_n, 0, sizeof(uint32_t) * NI, c->stream));
    // quotas: orb.cpp computeKeyPoints
    const float factor = (float)(1.0 / c->scale_factor);
    float ndes = c->cfg.n_features * (1 - factor) / (1 - (float)std::pow((double)factor, (double)L));
    std::vector<int> quota(L);
    int sum = 0;
    for (int l = 0; l < L - 1; ++l) { quota[l] = cv_round_f(ndes); sum += quota[l]; ndes *= factor; }
    quota[L - 1] = std::max(c->cfg.n_features - sum, 0);
    DetectParams p = detect_params(c);
    const bool harris = use_harris(c);
    const uint8_t *prev = b.img;
    int pw = g0.w, ph = g0.h, ppitch = g0.pitch;
    size_t pstride = g0.img_stride;
    std::vector<int> tab;
    for (int l = 0; l < L; ++l) {
        const float scale = (float)std::pow(c->scale_factor, (double)l);
        Geom gl = g0;
        Buffers v = b;
        if (l > 0) {
            const float inv = 1.f / scale;
            const int dw = cv_round_f(g0.w * inv), dh = cv_round_f(g0.h * inv);
            if (dw < 7 || dh < 7) break;                          // nothing can be detected on smaller levels
            // INTER_LINEAR_EXACT tables (resize.cpp interpolationLinear), same double arithmetic as the oracle
            tab.assign(2 * (size_t)(dw + dh), 0);
            auto fill = [&](int src, int dst, int *ofs, int *a1) {
                const double sc = 1.0 / ((double)dst / (double)src);
                for (int i = 0; i < dst; ++i) {
                    const double sf = sc * (i + 0.5) - 0.5;
                    const int si = (int)std::floor(sf);
                    if (si < 0) { ofs[i] = 0; a1[i] = 0; }
                    else if (si + 1 >= src) { ofs[i] = src - 1; a1[i] = 0; }
                    else { ofs[i] = si; a1[i] = (int)lrint((sf - si) * 256.0); }
                }
            };
            fill(pw, dw, tab.data(), tab.data() + dw);
            fill(ph, dh, tab.data() + 2 * dw, tab.data() + 2 * dw + dh);
            // the table of the previous level may still be in use by its resize kernel: stream order + a sync-free
            // staging would need two tables; levels are few, so synchronise before overwriting the pinned-less copy
            FE_CUDA(c, cudaStreamSynchronize(c->stream));
            FE_CUDA(c, cudaMemcpyAsync(b.pyr_tab, tab.data(), sizeof(int) * tab.size(), cudaMemcpyHostToDevice, c->stream));
            gl.w = dw; gl.h = dh; gl.pitch = round_up(dw, 16);
            set_strip_geometry(gl, c->cfg.nonmax != 0);
            gl.img_stride = (size_t)gl.pitch * dh;
            uint8_t *cur = (l & 1) ? b.pyr_img1 : b.pyr_img0;
            { StageTimer t(c, ST_BLUR);
              t.done(launch_resize_linear_exact(prev, pw, ph, ppitch, pstride, cur, dw, dh, gl.pitch, gl.img_stride, b.pyr_tab, NI, c->stream)); }
            v.img = cur;
            prev = cur; pw = dw; ph = dh; ppitch = gl.pitch; pstride = gl.img_stride;
        }
        if (harris && 2 * (long long)quota[l] > g0.kp_cap)
            return fail(c, FE_ERR_CAPACITY, "HARRIS_SCORE keeps 2 x quota FAST corners per level before the Harris cut: raise fe_config.max_keypoints");
        p.n_features = harris ? 2 * quota[l] : quota[l];
        { StageTimer t(c, ST_FAST); t.done(launch_fast(gl, p, v, c->stream)); }
        { StageTimer t(c, ST_SELECT); t.done(launch_select(gl, p, v, c->stream)); }
        if (harris) { StageTimer t(c, ST_SELECT); t.done(launch_harris_select(gl, quota[l], v, c->stream)); }
        { StageTimer t(c, ST_ORIENT); t.done(launch_orient(gl, p, v, true, c->stream)); }
        if (harris) { StageTimer t(c, ST_ORIENT); t.done(launch_harris_store(gl, v, c->stream)); }
        if (describe) {
            { StageTimer t(c, ST_BLUR); t.done(launch_blur(gl, v, c->stream)); }
            { StageTimer t(c, ST_BRIEF); t.done(launch_rbrief(gl, p, v, v.n_kp, c->stream)); }
        }
        { StageTimer t(c, ST_SELECT);
          t.done(launch_pyr_append(gl, l, scale, (float)c->patch_size * scale, v, b.pyr_kp, b.pyr_desc, b.pyr_n, describe, c->stream)); }
    }
    const size_t C = (size_t)g0.kp_cap;
    FE_CUDA(c, cudaMemcpyAsync(b.kp, b.pyr_kp, sizeof(fe_kpoint) * C * NI, cudaMemcpyDeviceToDevice, c->stream));
    if (describe) FE_CUDA(c, cudaMemcpyAsync(b.desc, b.pyr_desc, 32 * C * NI, cudaMemcpyDeviceToDevice, c->stream));
    FE_CUDA(c, cudaMemcpyAsync(b.n_kp, b.pyr_n, sizeof(uint32_t) * NI, cudaMemcpyDeviceToDevice, c->stream));
    { StageTimer t(c, ST_ORIENT); t.done(launch_pyr_coords(g0, b, c->stream)); }
    FE_CUDA(c, cudaGetLastError());
    return FE_OK;
}

int run_detect(fe_ctx *c, bool describe) {
    apply_pending_detection(c);
    if (c->nlevels > 1) return run_detect_pyramid(c, describe);
    return run_detect_on(c, c->g, c->b, c->stream, describe, true);
}

MatchParams match_params(const fe_match_cfg *a) {
    MatchParams mp{};
    mp.mask = a ? a->mask : FE_MASK_NONE;
    mp.epi_threshold = a ? a->epi_threshold : 0.f;
    mp.q_off = a ? a->q_y_offset : 0.f;
    mp.t_off = a ? a->t_y_offset : 0.f;
    mp.half_w = a ? (float)(a->win_w / 2) : 0.f;
    mp.half_h = a ? (float)(a->win_h / 2) : 0.f;
    mp.h2 = (a && a->norm == FE_NORM_HAMMING2) ? 1 : 0;
    return mp;
}

// What the matchers read beyond the core buffers: L2 keys for float descriptors (dim > 0), and mode B's scratch -- the
// tensor-core verification for L2, the pruned cross-check for Hamming.  Allocated before any view of the buffers is taken.
unsigned match_groups(int dim, bool cross) {
    if (dim > 0) return GRP_FLOAT | (cross ? GRP_VERIFY : 0u);
    return cross ? GRP_CROSS : 0u;
}

// Largest SURF window among the keypoints this ctx detects itself: size 7 for plain FAST keypoints, patchSize * scale^level
// in ORB mode (launch_pyr_append writes size = patch_size * scale), evaluated exactly like the kernel's win_size
int detected_surf_win(const fe_ctx *c) {
    float size = 7.f;
    if (c->cfg.orientation) size = (float)c->patch_size * (float)std::pow(c->scale_factor, (double)(c->nlevels - 1));
    return (int)(21.f * (size * 1.2f / 9.0f));
}

int desc_dim(int kind) { return kind == FE_DESC_SURF64 ? 64 : kind == FE_DESC_SURF128 ? 128 : 0; }
// cv::BriefDescriptorExtractor rows: bytes per descriptor (0 for the other kinds)
int brief_width(int kind) { return kind == FE_DESC_BRIEF16 ? 16 : kind == FE_DESC_BRIEF32 ? 32 : kind == FE_DESC_BRIEF64 ? 64 : 0; }
int brief_slot(int kind) { return kind - FE_DESC_BRIEF16; }
// Bytes of a binary row on the host, packed as fe_describe writes it: 16 for BRIEF-16, 32 for ORB-256 and BRIEF-32.  The
// matchers' device rows are 32 bytes; BRIEF-16 rows ride in them zero-padded, which leaves every Hamming distance unchanged.
int binary_bytes(int kind) { return kind == FE_DESC_BRIEF16 ? 16 : 32; }

// What rows the batch holds: SURF-64 / SURF-128 per fe_surf_params.extended when it detects with the Fast-Hessian detector,
// else what fe_set_batch_descriptor selected.
int batch_rows(const fe_ctx *c) { return c->hessian ? (c->surf.extended ? FE_DESC_SURF128 : FE_DESC_SURF64) : c->batch_desc; }
// Whether the SURF rows of the batch are upright (no orientation, no integral image for it)
bool batch_upright(const fe_ctx *c) { return c->hessian ? c->surf.upright != 0 : c->cfg.surf_upright != 0; }
// Whether every image's keypoints are in raster order: always with the Fast-Hessian detector, else without a pyramid (the
// pyramid's keypoints are level-major)
bool batch_raster(const fe_ctx *c) { return c->hessian || c->nlevels == 1; }

// (g, b, st): the batch -- or the chunk view of it -- to match; timed = false on the auxiliary streams of the chunked pipeline.
// Needs the groups of match_groups(dim, cfg_b != nullptr).
int run_match_l2_on(fe_ctx *c, const Geom &g, const Buffers &b, cudaStream_t st, bool timed, int n_pairs, int dim,
                    const fe_match_cfg *cfg_a, const fe_match_cfg *cfg_b, const uint32_t *counts, bool train_sorted) {
    const bool masked = cfg_a && cfg_a->mask != FE_MASK_NONE;
    const bool unmasked_knn = cfg_a && cfg_a->mask == FE_MASK_NONE;
    const bool want_all = cfg_b != nullptr;
    // Mode B with the |dy| post-filter on raster-ordered trains: band candidates + ONE tcgen05 GEMM + verification.  Exact.
    const bool verify = c->l2_tensor >= 1 && cfg_b && cfg_b->max_dy >= 0.f && train_sorted;
    if (verify) {
        // mode A's band pass visits a superset of mode B's band: let it produce the cross-check candidates as well
        const bool fuse = cfg_a && cfg_a->mask == FE_MASK_EPIPOLAR && cfg_a->q_y_offset == 0.f && cfg_a->t_y_offset == 0.f &&
                          cfg_a->epi_threshold >= cfg_b->max_dy;
        if (fuse) {
            StageTimer t(c, ST_L2, st, timed);
            t.done(launch_l2_band_cand(g, n_pairs, dim, match_params(cfg_a), cfg_b->max_dy, true, b, counts, st));
        } else {
            if (masked && train_sorted) { StageTimer t(c, ST_L2, st, timed); t.done(launch_l2_band(g, n_pairs, dim, match_params(cfg_a), b, counts, st)); }
            else if (cfg_a) { StageTimer t(c, ST_L2, st, timed); t.done(launch_l2_match(g, n_pairs, dim, match_params(cfg_a), true, false, b, counts, st)); }
            MatchParams mpb{};
            mpb.mask = FE_MASK_EPIPOLAR; mpb.epi_threshold = cfg_b->max_dy;
            StageTimer t(c, ST_L2, st, timed);
            t.done(launch_l2_band_cand(g, n_pairs, dim, mpb, cfg_b->max_dy, false, b, counts, st));
        }
        { StageTimer t(c, ST_L2AUX, st, timed); t.done(launch_l2_verify(g, n_pairs, dim, b, counts, 0, st)); }
        { StageTimer t(c, ST_L2TC, st, timed); t.done(launch_l2_verify(g, n_pairs, dim, b, counts, 1, st)); }
        { StageTimer t(c, ST_L2AUX, st, timed); t.done(launch_l2_verify(g, n_pairs, dim, b, counts, 2, st)); }
        FE_CUDA(c, cudaMemcpyAsync(c->h_tc_error, b.tc_error, sizeof(int), cudaMemcpyDeviceToHost, st));
    } else if (c->l2_tensor >= 2 && (want_all || unmasked_knn)) {
        // opt-in (FE_L2_TENSOR=2), APPROXIMATE: bf16 tcgen05 GEMM proposes candidates per row, FP32 re-rank decides among them;
        // a true neighbour outside the shortlist is lost (no error bound) -- kept for A/B measurements only
        { StageTimer t(c, ST_L2AUX, st, timed); t.done(launch_l2_tensor(g, n_pairs, dim, unmasked_knn, b, counts, 0, st)); }
        { StageTimer t(c, ST_L2TC, st, timed); t.done(launch_l2_tensor(g, n_pairs, dim, unmasked_knn, b, counts, 1, st)); }
        { StageTimer t(c, ST_L2AUX, st, timed); t.done(launch_l2_tensor(g, n_pairs, dim, unmasked_knn, b, counts, 2, st)); }
        FE_CUDA(c, cudaMemcpyAsync(c->h_tc_error, b.tc_error, sizeof(int), cudaMemcpyDeviceToHost, st));
        if (masked && train_sorted) { StageTimer t(c, ST_L2, st, timed); t.done(launch_l2_band(g, n_pairs, dim, match_params(cfg_a), b, counts, st)); }
        else if (masked) { StageTimer t(c, ST_L2, st, timed); t.done(launch_l2_match(g, n_pairs, dim, match_params(cfg_a), true, false, b, counts, st)); }
    } else if (masked && train_sorted && !want_all) {
        StageTimer t(c, ST_L2, st, timed);
        t.done(launch_l2_band(g, n_pairs, dim, match_params(cfg_a), b, counts, st));
    } else {
        StageTimer t(c, ST_L2, st, timed);
        t.done(launch_l2_match(g, n_pairs, dim, match_params(cfg_a), cfg_a != nullptr, want_all, b, counts, st));
    }
    { StageTimer t(c, ST_FINALIZE, st, timed);
      int n = 0;
      if (cfg_a) n += launch_l2_finalize_ratio(g, n_pairs, cfg_a->ratio, b, counts, st);
      if (cfg_b) n += launch_l2_finalize_cross(g, n_pairs, cfg_b->max_dy, b, counts, st);
      t.done(n); }
    FE_CUDA(c, cudaGetLastError());
    return FE_OK;
}

// train_sorted: the train keypoints of every pair are in raster order (y non-decreasing), which
// makes the mask-allowed trains of a query one contiguous index range (banded kernel).  row_bytes: binary_bytes of the rows.
// Needs the groups of match_groups(0, cfg_b != nullptr).
int run_match_on(fe_ctx *c, const Geom &g, const Buffers &b, cudaStream_t st, bool timed, int n_pairs,
                 const fe_match_cfg *cfg_a, const fe_match_cfg *cfg_b, const uint32_t *counts, bool train_sorted,
                 bool both_sorted, int row_bytes) {
    auto binary = [](const fe_match_cfg *m) { return !m || m->norm == FE_NORM_HAMMING || m->norm == FE_NORM_HAMMING2; };
    if (!binary(cfg_a) || !binary(cfg_b))
        return fail(c, FE_ERR_UNSUPPORTED, "binary descriptors are matched with FE_NORM_HAMMING or FE_NORM_HAMMING2");
    // Mode B with the |dy| post-filter on raster-ordered keypoints: band candidates + pruned verification (exact; about
    // half the instructions of the all-pairs kernel).  FE_CROSS_PRUNE=0 forces the all-pairs kernel (A/B testing).
    const bool pruned = cfg_b && c->cross_prune && both_sorted && cfg_b->norm == FE_NORM_HAMMING && cfg_b->max_dy >= 0.f;
    // mode A's band pass visits a superset of mode B's band: let it produce the cross-check candidates as well
    const bool fuse_band = pruned && cfg_a && train_sorted && cfg_a->norm == FE_NORM_HAMMING && cfg_a->mask == FE_MASK_EPIPOLAR &&
                           cfg_a->q_y_offset == 0.f && cfg_a->t_y_offset == 0.f && cfg_a->epi_threshold >= cfg_b->max_dy;
    if (cfg_a) {
        StageTimer t(c, ST_KNN, st, timed);
        t.done(launch_hamming_knn2(g, n_pairs, match_params(cfg_a), train_sorted, b, counts, fuse_band ? cfg_b->max_dy : -1.f, st));
    }
    if (cfg_b) {
        StageTimer t(c, ST_MATCH, st, timed);
        if (pruned) {
            // the join (latency / issue bound) runs on a side stream beside the verification scans (ALU / POPC bound); the stage's
            // events on `st` still bracket all of it
            const int lane = st == c->stream ? 0 : st == c->s_cmp[0] ? 1 : st == c->s_cmp[1] ? 2 : -1;
            static const bool overlap = !(getenv("FE_CX_OVERLAP") && atoi(getenv("FE_CX_OVERLAP")) == 0);      // A/B testing
            if (overlap && lane >= 0 && !c->s_aux[lane]) {
                FE_CUDA(c, cudaStreamCreateWithFlags(&c->s_aux[lane], cudaStreamNonBlocking));
                FE_CUDA(c, cudaEventCreateWithFlags(&c->ev_fork[lane], cudaEventDisableTiming));
                FE_CUDA(c, cudaEventCreateWithFlags(&c->ev_join[lane], cudaEventDisableTiming));
            }
            const bool side = overlap && lane >= 0;
            t.done(launch_hamming_cross_pruned(g, n_pairs, cfg_b->max_dy, fuse_band, c->cross_mih, row_bytes, b, counts, cfg_a ? std::max(cfg_a->ratio, 0.0) : -1.0, st,
                                               side ? c->s_aux[lane] : nullptr, side ? c->ev_fork[lane] : nullptr, side ? c->ev_join[lane] : nullptr));
        }
        else t.done(launch_hamming_cross(g, n_pairs, cfg_b->norm == FE_NORM_HAMMING2, b, counts, st));
    }
    {
        StageTimer t(c, ST_FINALIZE, st, timed);
        int n = 0;
        if (cfg_a && !(cfg_b && pruned)) n += launch_finalize_ratio(g, n_pairs, cfg_a->ratio, b, counts, st);    // (else: fused into the cross-check's finalize)
        if (cfg_b && !pruned) n += launch_finalize_cross(g, n_pairs, cfg_b->max_dy, b, counts, st);
        t.done(n);
    }
    FE_CUDA(c, cudaGetLastError());
    return FE_OK;
}

// Checks the match configs against the batch descriptor and allocates what run_batch_on reads beyond the core buffers.  Runs
// before any view of the buffers is taken, and its zero-fills are on the ctx stream.
int prepare_batch(fe_ctx *c, const fe_match_cfg *cfg_a, const fe_match_cfg *cfg_b) {
    const int dim = desc_dim(batch_rows(c));
    if (dim > 0 && ((cfg_a && cfg_a->norm != FE_NORM_L2) || (cfg_b && cfg_b->norm != FE_NORM_L2)))
        return fail(c, FE_ERR_UNSUPPORTED, "SURF descriptors are matched with FE_NORM_L2");
    const unsigned hessian = c->hessian ? GRP_INTEGRAL | GRP_SURFDET : 0u;      // the scale space reads the integral image
    const unsigned brief = brief_width(batch_rows(c)) > 0 && !batch_raster(c) ? GRP_INTEGRAL : 0u;   // brief_kernel's input
    return ensure(c, match_groups(dim, cfg_b != nullptr) | (dim > 0 && !batch_upright(c) ? GRP_INTEGRAL : 0u) | hessian | brief);
}

// cv::SURF's Fast-Hessian detector (src/surf.cpp:462-512) on the images of (g, b) in b.img: integral image, scale-space layers
// and maxima, HESSIAN_CHUNK_IMAGES images per pass through the one scale space of the ctx.  Leaves the unsorted maxima in
// b.hes_kp and their counts (which may exceed kp_cap) in b.hes_count.  max_win (optional): the largest descriptor window
// (int)(21 * size * 1.2 / 9) a keypoint of this layer schedule can have -- an interpolated maximum of a middle layer is no
// larger than the layer above it -- so that a caller can pick the descriptor variant without reading anything back.
// Needs GRP_INTEGRAL and GRP_SURFDET.  Used by fe_surf_detect_* and by the batched pipeline (fe_set_batch_detector).
int hessian_detect(fe_ctx *c, const Geom &g, const Buffers &b, const fe_surf_params *sp, cudaStream_t st, bool timed, int *max_win) {
    const int nOct = sp->n_octaves > 0 ? sp->n_octaves : 4, nLay = sp->n_octave_layers > 0 ? sp->n_octave_layers : 2;
    const int R = g.h, C = g.w, stride_i = g.w + 1;        // the integral image is (h + 1) x (w + 1)
    const int n_images = g.n_images;
    const size_t MI = c->cfg.max_images;
    // layer schedule
    const int nTotal = (nLay + 2) * nOct;
    std::vector<int> sizes(nTotal), steps(nTotal);
    std::vector<size_t> offs(nTotal + 1, 0);
    for (int o = 0, idx = 0, step = 1; o < nOct; ++o, step *= 2)
        for (int l = 0; l < nLay + 2; ++l, ++idx) {
            sizes[idx] = (9 + 6 * l) << o;
            steps[idx] = step;
            offs[idx + 1] = offs[idx] + (size_t)(R / step) * (size_t)(C / step);
        }
    const size_t per_image = (size_t)c->cfg.max_width * c->cfg.max_height * 10 * 2;     // floats of scale space per image (capacity)
    const int IC = std::min(c->cfg.max_images, HESSIAN_CHUNK_IMAGES);                       // images per scale-space chunk
    if (offs[nTotal] > per_image)
        return fail(c, FE_ERR_CAPACITY, "fe_surf_detect: too many octave layers for the scale-space buffer");
    { StageTimer t(c, ST_SURF, st, timed); t.done(launch_integral(g, b, st)); }
    FE_CUDA(c, cudaMemsetAsync(b.hes_count, 0, sizeof(uint32_t) * 2 * MI, st));
    static const int DX[3][5] = {{0, 2, 3, 7, 1}, {3, 2, 6, 7, -2}, {6, 2, 9, 7, 1}};
    static const int DY[3][5] = {{2, 0, 7, 3, 1}, {2, 3, 7, 6, -2}, {2, 6, 7, 9, 1}};
    static const int DXY[4][5] = {{1, 1, 4, 4, 1}, {5, 1, 8, 4, -1}, {1, 5, 4, 8, -1}, {5, 5, 8, 8, 1}};
    auto resize_box = [](const int *src, int size) {      // resizeHaarPattern, src/surf.cpp:136-152
        const float ratio = (float)size / 9;
        HaarBoxI o;
        o.dx1 = cv_round_f(ratio * src[0]); o.dy1 = cv_round_f(ratio * src[1]);
        o.dx2 = cv_round_f(ratio * src[2]); o.dy2 = cv_round_f(ratio * src[3]);
        o.w = src[4] / ((float)(o.dx2 - o.dx1) * (o.dy2 - o.dy1));
        return o;
    };
    const size_t s_img = (size_t)(g.h + 1) * (g.w + 1);
    int win = 1;
    for (int c0 = 0; c0 < n_images; c0 += IC) {
        const int ic = std::min(IC, n_images - c0);
        {
            StageTimer t(c, ST_FAST, st, timed);
            int nl = 0;
            for (int i = 0; i < nTotal; ++i) {
                HessianLayer hl{};
                hl.size = sizes[i]; hl.step = steps[i];
                hl.valid = !(sizes[i] > R || sizes[i] > C);
                hl.samples_i = hl.valid ? 1 + (R - sizes[i]) / steps[i] : 0;
                hl.samples_j = hl.valid ? 1 + (C - sizes[i]) / steps[i] : 0;
                hl.margin = (sizes[i] / 2) / steps[i];
                for (int k = 0; k < 3; ++k) { hl.box[k] = resize_box(DX[k], sizes[i]); hl.box[3 + k] = resize_box(DY[k], sizes[i]); }
                for (int k = 0; k < 4; ++k) hl.box[6 + k] = resize_box(DXY[k], sizes[i]);
                nl += launch_hessian_layer(b.integral + (size_t)c0 * s_img, s_img, stride_i, R, C, hl, b.hes_det + offs[i], b.hes_trace + offs[i],
                                           per_image, ic, st);
            }
            t.done(nl);
        }
        {
            StageTimer t(c, ST_SELECT, st, timed);
            int nl = 0;
            for (int o = 0; o < nOct; ++o)
                for (int l = 1; l <= nLay; ++l) {
                    const int idx = o * (nLay + 2) + l, step = steps[idx];
                    const int rows = R / step, cols = C / step;
                    const int margin = (sizes[idx + 1] / 2) / step + 1;
                    const int n = launch_hessian_maxima(b.hes_det + offs[idx - 1], b.hes_det + offs[idx], b.hes_det + offs[idx + 1],
                                                        b.hes_trace + offs[idx], per_image, rows, cols, margin, sizes[idx], sizes[idx - 1],
                                                        step, o, sp->hessian_threshold, b.hes_kp + (size_t)c0 * g.kp_cap, g.kp_cap,
                                                        b.hes_count + c0, ic, st);
                    if (n) win = std::max(win, (int)(21.f * ((float)sizes[idx + 1] * 1.2f / 9.0f)));
                    nl += n;
                }
            t.done(nl);
        }
    }
    if (max_win) *max_win = win;
    return FE_OK;
}

// cv::BriefDescriptorExtractor::compute (kind BRIEF-16 / 32 / 64) of the keypoints the detector left in (g, b), with the table
// and use_orientation set for that width now: runByImageBorder(28) on the device, then the rows, row_bytes apart, into out.
// Raster-ordered keypoints take the tile kernel, the pyramid's level-major ones brief_kernel over the integral images
// (GRP_INTEGRAL).  The caller checked that the table exists.
int run_brief_on(fe_ctx *c, const Geom &g, const Buffers &b, cudaStream_t st, bool timed, int kind, bool raster, uint8_t *out,
                 int row_bytes) {
    const int slot = brief_slot(kind), bw = brief_width(kind);
    const int8_t *tab = b.brief_tab + (size_t)slot * 512 * 4;
    // (timed as description: the border is compute()'s runByImageBorder, and fe_stereo_features reports it with the rows)
    { StageTimer t(c, ST_BRIEF, st, timed); t.done(launch_brief_border(g, b, st)); }
    if (raster) {
        StageTimer t(c, ST_BRIEF, st, timed);
        t.done(launch_brief_tile(g, b, tab, bw, c->brief_orient[slot], out, row_bytes, st));
    } else {
        { StageTimer t(c, ST_BLUR, st, timed); t.done(launch_integral(g, b, st)); }
        { StageTimer t(c, ST_BRIEF, st, timed); t.done(launch_brief_ext(g, b, b.n_kp, tab, bw, c->brief_orient[slot], out, row_bytes, st)); }
    }
    FE_CUDA(c, cudaGetLastError());
    return FE_OK;
}

// Detect, describe and match the batch (g, b) on st: the resident batch, or a chunk view of it.  ORB-256 or BRIEF-16 / 32 with
// Hamming matching, or FAST / ORB-mode keypoints with SURF descriptors (bin/detect_node:33-41) and L2 matching.  The caller applies
// pending detection changes and calls prepare_batch; the pyramid (nlevels > 1) runs on the whole resident batch only.
int run_batch_on(fe_ctx *c, const Geom &g, const Buffers &b, cudaStream_t st, bool timed, int n_pairs,
                 const fe_match_cfg *cfg_a, const fe_match_cfg *cfg_b) {
    const int rows = batch_rows(c), dim = desc_dim(rows);
    const bool sorted = batch_raster(c), brief = brief_width(rows) > 0;
    if (c->hessian) {
        // Fast-Hessian maxima -> the survivors in raster order -> descriptors; nothing returns to the host
        int max_win = 0;
        int r = hessian_detect(c, g, b, &c->surf, st, timed, &max_win);
        if (r != FE_OK) return r;
        { StageTimer t(c, ST_SELECT, st, timed); t.done(launch_surf_raster(g, b.hes_kp, b.hes_count, batch_upright(c), b, st)); }
        { StageTimer t(c, ST_SURF, st, timed); t.done(launch_surf(g, b, b.n_kp, dim == 128, batch_upright(c), max_win, st)); }
    } else {
        const bool orb = dim == 0 && !brief;
        int r = sorted ? run_detect_on(c, g, b, st, orb, timed) : run_detect_pyramid(c, orb);
        if (r != FE_OK) return r;
        if (dim > 0) {
            StageTimer t(c, ST_SURF, st, timed);
            t.done(launch_surf(g, b, b.n_kp, dim == 128, batch_upright(c), detected_surf_win(c), st));
        }
        if (brief && (r = run_brief_on(c, g, b, st, timed, rows, sorted, b.desc, 32)) != FE_OK) return r;
    }
    if (!cfg_a && !cfg_b) return FE_OK;
    if (dim > 0) return run_match_l2_on(c, g, b, st, timed, n_pairs, dim, cfg_a, cfg_b, b.n_kp, sorted);
    return run_match_on(c, g, b, st, timed, n_pairs, cfg_a, cfg_b, b.n_kp, sorted, sorted, binary_bytes(rows));
}

// Counts of pairs [p0, p0 + np) into h_counts: keypoints of image i at [i], n_a of pair p at [NI + p], n_b at [NI + NP + p]
// (NI images, NP pairs resident).
int copy_counts(fe_ctx *c, int p0, int np, cudaStream_t st) {
    const int NI = c->g.n_images, NP = NI / 2;
    uint32_t *hc = c->h_counts;
    FE_CUDA(c, cudaMemcpyAsync(hc + 2 * p0, c->b.n_kp + 2 * p0, sizeof(uint32_t) * 2 * np, cudaMemcpyDeviceToHost, st));
    FE_CUDA(c, cudaMemcpyAsync(hc + NI + p0, c->b.n_a + p0, sizeof(uint32_t) * np, cudaMemcpyDeviceToHost, st));
    FE_CUDA(c, cudaMemcpyAsync(hc + NI + NP + p0, c->b.n_b + p0, sizeof(uint32_t) * np, cudaMemcpyDeviceToHost, st));
    return FE_OK;
}

// Host arrays of a whole batch: kp_cap keypoints / descriptors per image and matches per pair; null arrays are skipped.
struct HostBatch {
    int32_t kp_cap;
    fe_kpoint *kps;
    uint8_t *desc;
    int32_t *n_kps;
    fe_match *ma;
    int32_t *n_a;
    fe_match *mb;
    int32_t *n_b;
};

// Downloads pairs [p0, p0 + np) of the resident batch on st into o, sized by the counts copy_counts left in h_counts:
// reports the counts, sets `overflow` if a keypoint count exceeds either capacity, accounts the bytes and copies the used
// prefix of every array, one strided copy per array (rows = images or pairs).
int download_pairs(fe_ctx *c, int p0, int np, cudaStream_t st, const HostBatch &o, bool &overflow) {
    const Geom &g = c->g;
    const int NI = g.n_images, NP = NI / 2, i0 = 2 * p0, ni = 2 * np, cap = o.kp_cap;
    const uint32_t *hc = c->h_counts;
    int max_kp = 0, max_a = 0, max_b = 0;
    for (int i = i0; i < i0 + ni; ++i) {
        if ((int)hc[i] > cap || (int)hc[i] > g.kp_cap) overflow = true;
        max_kp = std::max(max_kp, std::min(std::min((int)hc[i], cap), g.kp_cap));
        if (o.n_kps) o.n_kps[i] = (int32_t)hc[i];
    }
    for (int p = p0; p < p0 + np; ++p) {
        max_a = std::max(max_a, std::min((int)hc[NI + p], cap));
        max_b = std::max(max_b, std::min((int)hc[NI + NP + p], cap));
        if (o.n_a) o.n_a[p] = (int32_t)hc[NI + p];
        if (o.n_b) o.n_b[p] = (int32_t)hc[NI + NP + p];
    }
    const int rows = batch_rows(c), dim = desc_dim(rows);
    const size_t drow = dim > 0 ? sizeof(float) * dim : binary_bytes(rows);      // descriptor bytes per keypoint on the host
    const size_t dev_row = dim > 0 ? sizeof(float) * 128 : 32;                    // and on the device
    c->d2h_bytes += (int64_t)sizeof(uint32_t) * 2 * ni + (o.kps ? (int64_t)sizeof(fe_kpoint) * max_kp * ni : 0) +
                    (o.desc ? (int64_t)drow * max_kp * ni : 0) + (o.ma ? (int64_t)sizeof(fe_match) * max_a * np : 0) +
                    (o.mb ? (int64_t)sizeof(fe_match) * max_b * np : 0);
    const Buffers v = view_of(c->b, g, i0);
    const size_t C = g.kp_cap, K = cap;
    if (o.kps && max_kp > 0)
        FE_CUDA(c, cudaMemcpy2DAsync(o.kps + i0 * K, sizeof(fe_kpoint) * K, v.kp, sizeof(fe_kpoint) * C, sizeof(fe_kpoint) * max_kp,
                                     ni, cudaMemcpyDeviceToHost, st));
    const uint8_t *dsrc = dim ? reinterpret_cast<const uint8_t *>(v.fdesc) : v.desc;
    if (o.desc && max_kp > 0 && drow == dev_row)     // host rows as on the device (32 bytes or 128 floats): one strided copy
        FE_CUDA(c, cudaMemcpy2DAsync(o.desc + i0 * K * drow, drow * K, dsrc, drow * C, drow * max_kp, ni, cudaMemcpyDeviceToHost, st));
    if (o.desc && max_kp > 0 && drow < dev_row)      // SURF-64, BRIEF-16: pack the leading drow bytes of every device row
        for (int i = 0; i < ni; ++i)
            FE_CUDA(c, cudaMemcpy2DAsync(o.desc + (i0 + i) * K * drow, drow, dsrc + i * C * dev_row, dev_row, drow,
                                         std::min((int)hc[i0 + i], max_kp), cudaMemcpyDeviceToHost, st));
    if (o.ma && max_a > 0)
        FE_CUDA(c, cudaMemcpy2DAsync(o.ma + p0 * K, sizeof(fe_match) * K, v.match_a, sizeof(fe_match) * C, sizeof(fe_match) * max_a,
                                     np, cudaMemcpyDeviceToHost, st));
    if (o.mb && max_b > 0)
        FE_CUDA(c, cudaMemcpy2DAsync(o.mb + p0 * K, sizeof(fe_match) * K, v.match_b, sizeof(fe_match) * C, sizeof(fe_match) * max_b,
                                     np, cudaMemcpyDeviceToHost, st));
    return FE_OK;
}

// Reads and clears the tcgen05 completion-barrier flag that the L2 tensor-core matchers copy to the host (the streams they
// ran on must be synchronised).
bool take_tc_error(fe_ctx *c) {
    if (!*c->h_tc_error) return false;
    *c->h_tc_error = 0;
    cudaMemsetAsync(c->b.tc_error, 0, sizeof(int), c->stream);
    return true;
}

int sync_and_resolve(fe_ctx *c) {
    FE_CUDA(c, cudaStreamSynchronize(c->stream));
    resolve_pending(c);
    if (take_tc_error(c)) return fail(c, FE_ERR_CUDA, "l2_tensor: tcgen05 completion barrier timed out");
    return FE_OK;
}

}  // namespace

extern "C" {

int32_t fe_abi_version(void) { return FE_ABI_VERSION; }

int32_t fe_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

const char *fe_last_error(const fe_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

static int upload_orb_pattern(fe_ctx *c, int patch_size, int wta_k);

void fe_default_config(fe_config *cfg) {
    if (!cfg) return;
    *cfg = fe_config{};
    cfg->max_width = 1920; cfg->max_height = 1200; cfg->max_images = 2; cfg->max_keypoints = 16384;
    cfg->fast_threshold = 15; cfg->fast_type = FE_FAST_9_16; cfg->nonmax = 1; cfg->n_features = 5000;
    cfg->edge_threshold = 31; cfg->orientation = 1; cfg->surf_upright = 1;
}

int32_t fe_create(const fe_config *cfg_in, fe_ctx **out) {
    if (!out) return FE_ERR_BAD_ARG;
    *out = nullptr;
    fe_config cfg{};
    if (cfg_in) cfg = *cfg_in;
    if (cfg.max_width <= 0) cfg.max_width = 1920;
    if (cfg.max_height <= 0) cfg.max_height = 1200;
    if (cfg.max_images <= 0) cfg.max_images = 2;
    if (cfg.max_keypoints <= 0) cfg.max_keypoints = 16384;
    if (cfg.fast_threshold <= 0) cfg.fast_threshold = 15;
    if (cfg.fast_type == 0) cfg.fast_type = FE_FAST_9_16;
    if (cfg_in == nullptr) { cfg.nonmax = 1; cfg.n_features = 5000; cfg.edge_threshold = 31; cfg.orientation = 1; }
    if (cfg.max_keypoints > 65535) { g_create_error = "max_keypoints must be <= 65535"; return FE_ERR_BAD_ARG; }
    if (cfg.fast_type != 16 && cfg.fast_type != 12 && cfg.fast_type != 8) {
        g_create_error = "fast_type must be 16, 12 or 8"; return FE_ERR_BAD_ARG;
    }
    if (cfg.edge_threshold < 0 || cfg.max_width > 16384) { g_create_error = "bad edge_threshold/max_width"; return FE_ERR_BAD_ARG; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        g_create_error = "no CUDA device available (this library has no CPU fallback)";
        return FE_ERR_NO_DEVICE;
    }
    if (cfg.device < 0 || cfg.device >= ndev) { g_create_error = "bad device ordinal"; return FE_ERR_BAD_ARG; }
    fe_ctx *c = new fe_ctx();
    c->cfg = cfg;
    if (const char *e = getenv("FE_L2_TENSOR")) c->l2_tensor = atoi(e);
    if (const char *e = getenv("FE_CROSS_PRUNE")) c->cross_prune = atoi(e) != 0;
    if (const char *e = getenv("FE_CROSS_MIH")) c->cross_mih = atoi(e) != 0;
    auto bail = [&](cudaError_t e, const char *what) {
        g_create_error = std::string(what) + ": " + cudaGetErrorString(e);
        fe_destroy(c);
        return (int32_t)FE_ERR_CUDA;
    };
    cudaError_t e;
    if ((e = cudaSetDevice(cfg.device)) != cudaSuccess) return bail(e, "cudaSetDevice");
    if (cfg.stream) c->stream = (cudaStream_t)cfg.stream;
    else {
        if ((e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(e, "cudaStreamCreate");
        c->own_stream = true;
    }
    c->gmax = geom_of(cfg, cfg.max_width, cfg.max_height, cfg.max_images);
    if (ensure(c, GRP_CORE) != FE_OK) { g_create_error = c->err; fe_destroy(c); return FE_ERR_CUDA; }
    if ((e = cudaHostAlloc(reinterpret_cast<void **>(&c->h_counts), sizeof(uint32_t) * 3 * cfg.max_images, cudaHostAllocDefault)) != cudaSuccess ||
        (e = cudaHostAlloc(reinterpret_cast<void **>(&c->h_tc_error), sizeof(int), cudaHostAllocDefault)) != cudaSuccess)
        return bail(e, "cudaHostAlloc");
    *c->h_tc_error = 0;
    if ((e = cudaStreamSynchronize(c->stream)) != cudaSuccess) return bail(e, "cudaStreamSynchronize");
    if (upload_orb_pattern(c, 31, 2) != FE_OK) { g_create_error = c->err; fe_destroy(c); return FE_ERR_CUDA; }
    *out = c;
    return FE_OK;
}

void fe_destroy(fe_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->cfg.device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    for_each_buffer(c->b, c->gmax, [](auto *&p, size_t, BufScope, unsigned, const char *) { if (p) cudaFree(p); });
    if (c->h_counts) cudaFreeHost(c->h_counts);
    if (c->h_tc_error) cudaFreeHost(c->h_tc_error);
    for (auto &p : c->pending) { cudaEventDestroy(p.a); cudaEventDestroy(p.b); }
    for (auto e : c->pool) cudaEventDestroy(e);
    for (auto e : c->ev_in) cudaEventDestroy(e);
    for (auto e : c->ev_done) cudaEventDestroy(e);
    if (c->ev_sync) cudaEventDestroy(c->ev_sync);
    for (cudaStream_t st : {c->s_in, c->s_out, c->s_cmp[0], c->s_cmp[1]}) if (st) cudaStreamDestroy(st);
    for (int i = 0; i < 3; ++i) {
        if (c->s_aux[i]) cudaStreamDestroy(c->s_aux[i]);
        if (c->ev_fork[i]) cudaEventDestroy(c->ev_fork[i]);
        if (c->ev_join[i]) cudaEventDestroy(c->ev_join[i]);
    }
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

int32_t fe_set_detection(fe_ctx *c, int32_t threshold, int32_t set_point, int32_t *new_set_point) {
    if (!c) return FE_ERR_BAD_ARG;
    if (threshold < 1 || threshold > 255) return fail(c, FE_ERR_BAD_ARG, "threshold must be in [1,255]");
    c->pending_threshold.store(threshold);
    c->pending_setpoint.store(set_point);
    if (new_set_point) *new_set_point = set_point;   // res.newSetPoint = setPoint (live_stereo.cpp:110)
    return FE_OK;
}

int32_t fe_sync(fe_ctx *c) {
    if (!c) return FE_ERR_BAD_ARG;
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    return sync_and_resolve(c);
}

void *fe_stream(fe_ctx *c) { return c ? (void *)c->stream : nullptr; }

void *fe_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}

void fe_host_free(void *p) { if (p) cudaFreeHost(p); }

int32_t fe_profile_enable(fe_ctx *c, int32_t on) {
    if (!c) return FE_ERR_BAD_ARG;
    c->profiling = on != 0;
    return FE_OK;
}

int32_t fe_profile_reset(fe_ctx *c) {
    if (!c) return FE_ERR_BAD_ARG;
    int r = sync_and_resolve(c);
    for (int i = 0; i < ST_COUNT; ++i) { c->stage_ms[i] = 0; c->stage_launches[i] = 0; }
    return r;
}

int32_t fe_stage_times(fe_ctx *c, int32_t cap, const char **names, double *ms, int64_t *launches, int32_t *n_stages) {
    if (!c) return FE_ERR_BAD_ARG;
    int r = sync_and_resolve(c);
    if (r != FE_OK) return r;
    if (n_stages) *n_stages = ST_COUNT;
    for (int i = 0; i < ST_COUNT && i < cap; ++i) {
        if (names) names[i] = kStageNames[i];
        if (ms) ms[i] = c->stage_ms[i];
        if (launches) launches[i] = c->stage_launches[i];
    }
    return FE_OK;
}

int64_t fe_kernel_launches(const fe_ctx *c) { return c ? c->launches : 0; }

int32_t fe_transfer_bytes(const fe_ctx *c, int64_t *h2d, int64_t *d2h) {
    if (!c) return FE_ERR_BAD_ARG;
    if (h2d) *h2d = c->h2d_bytes;
    if (d2h) *d2h = c->d2h_bytes;
    return FE_OK;
}

// POPC-pipe peak: the denominator of the Hamming matcher's roofline, measured on this device by a
// register-only kernel (8 independent POPC chains per thread, no memory traffic).
int32_t fe_measure_popc_peak(fe_ctx *c, double *gpopc_per_s) {
    if (!c || !gpopc_per_s) return FE_ERR_BAD_ARG;
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    cudaEvent_t e0, e1;
    FE_CUDA(c, cudaEventCreate(&e0));
    FE_CUDA(c, cudaEventCreate(&e1));
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->cfg.device);
    const int iters = 4096;
    double best_ms = 1e30;
    double ops = 0;
    for (int rep = 0; rep < 4; ++rep) {
        cudaEventRecord(e0, c->stream);
        ops = launch_popc_peak(sms, iters, c->b.allbest, c->stream);
        cudaEventRecord(e1, c->stream);
        FE_CUDA(c, cudaStreamSynchronize(c->stream));
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (rep > 0 && ms < best_ms) best_ms = ms;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *gpopc_per_s = ops / (best_ms * 1e-3) / 1e9;
    return FE_OK;
}

// ---- single-image primitives ----------------------------------------------------------------------

int32_t fe_detect(fe_ctx *c, const uint8_t *img, int32_t w, int32_t h, int32_t stride, fe_kpoint *out,
                  int32_t cap, int32_t *n) {
    if (!c || !img || !n || cap < 0 || (cap > 0 && !out) || stride < w) return fail(c, FE_ERR_BAD_ARG, "fe_detect: bad argument");
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    int r = set_geom(c, w, h, 1);
    if (r != FE_OK) return r;
    { StageTimer t(c, ST_H2D); r = upload_images(c, img, 1, stride, 0, 1); t.done(0); }
    if (r != FE_OK) return r;
    if ((r = run_detect(c, false)) != FE_OK) return r;
    FE_CUDA(c, cudaMemcpyAsync(c->h_counts, c->b.n_kp, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    FE_CUDA(c, cudaStreamSynchronize(c->stream));
    const int found = (int)c->h_counts[0];
    *n = found;
    const int m = std::min(std::min(found, cap), c->g.kp_cap);
    if (m > 0) FE_CUDA(c, cudaMemcpyAsync(out, c->b.kp, sizeof(fe_kpoint) * m, cudaMemcpyDeviceToHost, c->stream));
    if ((r = sync_and_resolve(c)) != FE_OK) return r;
    if (found > cap || found > c->g.kp_cap) return fail(c, FE_ERR_CAPACITY, "fe_detect: more keypoints than capacity");
    return FE_OK;
}

// ---- grid detector with per-cell setpoint controller + cornerSubPix (live nodes) --------------------
// src/live_stereo.cpp:277-352 (variant 0) and src/front_end/features.py:609-641 (variant 1), one eye per call.
int32_t fe_grid_detect(fe_ctx *c, const uint8_t *img, int32_t w, int32_t h, int32_t stride, const fe_grid_cfg *gc,
                       int32_t *thresholds, fe_kpoint *out, int32_t cap, int32_t *n, int32_t *cell_counts) {
    if (!c || !img || !gc || !thresholds || !n || cap < 0 || (cap > 0 && !out) || stride < w)
        return fail(c, FE_ERR_BAD_ARG, "fe_grid_detect: bad argument");
    const int rows = gc->rows > 0 ? gc->rows : 2, cols = gc->cols > 0 ? gc->cols : 3, nc = rows * cols;
    const int ps = gc->fast_type ? gc->fast_type : FE_FAST_7_12;
    if (ps != 16 && ps != 12 && ps != 8) return fail(c, FE_ERR_BAD_ARG, "fe_grid_detect: fast_type must be 16, 12 or 8");
    if (nc > SUBPIX_MAX_IMAGES || nc > c->cfg.max_images)
        return fail(c, FE_ERR_CAPACITY, "fe_grid_detect: rows*cols exceeds min(16, fe_config.max_images)");
    if (w > c->cfg.max_width || h > c->cfg.max_height) return fail(c, FE_ERR_BAD_ARG, "image larger than fe_config.max_width/max_height");
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    const bool py = gc->variant == 1;
    const int rx = gc->roi_w > 0 ? gc->roi_x : 0, ry = gc->roi_w > 0 ? gc->roi_y : 0;
    const int rw = gc->roi_w > 0 ? gc->roi_w : w, rh = gc->roi_h > 0 ? gc->roi_h : h;
    // cell rectangles (full-image coordinates)
    int cw, ch, x_end, y_end;
    if (py) {   // features.py:610-620: roi w / h are END coordinates of the slice [y : h + 1, x : w + 1]
        cw = (int)((double)rw / cols); ch = (int)((double)rh / rows);
        x_end = std::min(rw + 1, w); y_end = std::min(rh + 1, h);
    } else {    // live_stereo.cpp:150-153
        cw = rw / cols; ch = rh / rows;
        x_end = std::min(rx + rw, w); y_end = std::min(ry + rh, h);
    }
    if (cw < 7 || ch < 7) return fail(c, FE_ERR_BAD_ARG, "fe_grid_detect: cells smaller than 7 x 7");
    if (rx < 0 || ry < 0 || rx + cols * cw > x_end || ry + rows * ch > y_end)
        return fail(c, FE_ERR_UNSUPPORTED, "fe_grid_detect: ROI cells must lie inside the image (equal-size cells only)");
    int r = set_geom(c, cw, ch, nc);
    if (r != FE_OK) return r;
    apply_pending_detection(c);
    const Geom &g = c->g;
    const int full_pitch = round_up(w, 16);
    {
        StageTimer t(c, ST_H2D);
        for (int k = 0; k < nc; ++k) {
            const int x0 = rx + (k % cols) * cw, y0 = ry + (k / cols) * ch;
            FE_CUDA(c, cudaMemcpy2DAsync(c->b.img + (size_t)k * g.img_stride, g.pitch, img + (size_t)y0 * stride + x0, stride,
                                         cw, ch, cudaMemcpyHostToDevice, c->stream));
        }
        if (py && gc->subpix)   // Python refines on the full rectified image
            FE_CUDA(c, cudaMemcpy2DAsync(c->b.blur, full_pitch, img, stride, w, h, cudaMemcpyHostToDevice, c->stream));
        for (int k = 0; k < nc; ++k) c->h_counts[k] = (uint32_t)std::max(thresholds[k], 1);
        FE_CUDA(c, cudaMemcpyAsync(c->b.thr_img, c->h_counts, sizeof(int) * nc, cudaMemcpyHostToDevice, c->stream));
        t.done(0);
    }
    DetectParams p;
    p.threshold = 0; p.ps = ps; p.nonmax = 1; p.n_features = -1; p.edge = 0; p.patch_size = c->patch_size; p.wta_k = c->wta_k;
    p.thr_img = c->b.thr_img;
    { StageTimer t(c, ST_FAST); t.done(launch_fast(g, p, c->b, c->stream)); }
    { StageTimer t(c, ST_SELECT); t.done(launch_select(g, p, c->b, c->stream)); }
    { StageTimer t(c, ST_ORIENT); t.done(launch_orient(g, p, c->b, false, c->stream)); }
    SubpixParams sp{};
    for (int k = 0; k < nc; ++k) {
        const int cx = (k % cols) * cw, cy = (k / cols) * ch;       // gridROI.x / .y (relative to the ROI)
        if (py) {
            sp.src[k] = c->b.blur; sp.w[k] = w; sp.h[k] = h; sp.pitch[k] = full_pitch;
            sp.pre_x[k] = (float)(cx + rx); sp.pre_y[k] = (float)(cy + ry);     // d.pt + xOffset + self.x, then refine
        } else {
            sp.src[k] = c->b.img + (size_t)k * g.img_stride; sp.w[k] = cw; sp.h[k] = ch; sp.pitch[k] = g.pitch;
            sp.post1_x[k] = (float)cx; sp.post1_y[k] = (float)cy;               // + gridROI, then + lroi
            sp.post2_x[k] = (float)rx; sp.post2_y[k] = (float)ry;
        }
    }
    sp.refine = gc->subpix ? 1 : 0; sp.max_iters = 40; sp.epsilon = 0.001f;
    { StageTimer t(c, ST_ORIENT); t.done(launch_subpix(g, c->b, c->b.n_kp, sp, c->stream)); }
    FE_CUDA(c, cudaGetLastError());
    FE_CUDA(c, cudaMemcpyAsync(c->h_counts, c->b.n_kp, sizeof(uint32_t) * nc, cudaMemcpyDeviceToHost, c->stream));
    FE_CUDA(c, cudaStreamSynchronize(c->stream));
    int total = 0, written = 0;
    bool overflow = false;
    std::vector<int> counts(nc);
    for (int k = 0; k < nc; ++k) {
        counts[k] = (int)c->h_counts[k];
        if (cell_counts) cell_counts[k] = counts[k];
        if (counts[k] > g.kp_cap) overflow = true;
        const int have = std::min(counts[k], g.kp_cap);
        const int m = std::min(have, cap - written);
        if (m > 0)
            FE_CUDA(c, cudaMemcpyAsync(out + written, c->b.kp + (size_t)k * g.kp_cap, sizeof(fe_kpoint) * m,
                                       cudaMemcpyDeviceToHost, c->stream));
        written += std::max(m, 0);
        total += counts[k];
    }
    *n = total;
    if ((r = sync_and_resolve(c)) != FE_OK) return r;
    if (gc->update) {
        // controller: live_stereo.cpp:84-102,294-318 / features.py:604-608,626-636
        const int lo = gc->min_threshold > 0 ? gc->min_threshold : (py ? 6 : 4), hi = gc->max_threshold > 0 ? gc->max_threshold : 80;
        const int bucket = py ? (int)((double)gc->set_point / (double)(rows * cols)) : (int)((float)gc->set_point / ((float)rows * cols));
        for (int k = 0; k < nc; ++k) {
            const double target = py ? ((k / cols) == 1 ? 2.0 * bucket : 0.5 * bucket) : (double)bucket;
            const double err = (double)counts[k] - target;
            if (std::fabs(err) > 0.2 * target) {
                const int t = thresholds[k] + (err > 0 ? 1 : -1);
                thresholds[k] = std::min(std::max(t, lo), hi);
            }
        }
    }
    if (overflow || total > cap) return fail(c, FE_ERR_CAPACITY, "fe_grid_detect: more keypoints than capacity");
    return FE_OK;
}

// cv::cornerSubPix(img, pts, Size(5,5), Size(-1,-1), TermCriteria(EPS + ITER, 40, 0.001)) for caller-supplied points
int32_t fe_corner_subpix(fe_ctx *c, const uint8_t *img, int32_t w, int32_t h, int32_t stride, fe_kpoint *kps, int32_t n) {
    if (!c || !img || (n > 0 && !kps) || n < 0 || stride < w) return fail(c, FE_ERR_BAD_ARG, "fe_corner_subpix: bad argument");
    if (n == 0) return FE_OK;
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    int r = set_geom(c, w, h, 1);
    if (r != FE_OK) return r;
    if (n > c->g.kp_cap) return fail(c, FE_ERR_CAPACITY, "more keypoints than fe_config.max_keypoints");
    for (int i = 0; i < n; ++i)
        if (!(kps[i].x >= 0.f && kps[i].x < (float)w && kps[i].y >= 0.f && kps[i].y < (float)h))
            return fail(c, FE_ERR_BAD_ARG, "fe_corner_subpix: point outside the image (cv::cornerSubPix asserts)");
    { StageTimer t(c, ST_H2D); r = upload_images(c, img, 1, stride, 0, 1); t.done(0); }
    if (r != FE_OK) return r;
    FE_CUDA(c, cudaMemcpyAsync(c->b.kp, kps, sizeof(fe_kpoint) * n, cudaMemcpyHostToDevice, c->stream));
    c->h_counts[0] = (uint32_t)n;
    FE_CUDA(c, cudaMemcpyAsync(c->b.n_override, c->h_counts, sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
    SubpixParams sp{};
    sp.src[0] = c->b.img; sp.w[0] = w; sp.h[0] = h; sp.pitch[0] = c->g.pitch;
    sp.refine = 1; sp.max_iters = 40; sp.epsilon = 0.001f;
    { StageTimer t(c, ST_ORIENT); t.done(launch_subpix(c->g, c->b, c->b.n_override, sp, c->stream)); }
    FE_CUDA(c, cudaGetLastError());
    FE_CUDA(c, cudaMemcpyAsync(kps, c->b.kp, sizeof(fe_kpoint) * n, cudaMemcpyDeviceToHost, c->stream));
    return sync_and_resolve(c);
}

// ---- cv::SURF::operator()(img, mask, kps, desc, useProvidedKeypoints = false): Fast-Hessian detector + descriptors ----
// src/surf.cpp:896-980 (driver), :462-512 (detector); selected by the detector table as "SURF" (features.py:149-156).
// Batched and device-resident: scale space, maxima, KeypointGreater sort, orientation + descriptors all stay on the device
// for n_images images; the only host round trip before the results is the count / largest-size read that sizes them.
static int surf_detect_impl(fe_ctx *c, int n_images, const uint8_t *imgs, int w, int h, int stride, const fe_surf_params *sp,
                            fe_kpoint *kps, float *desc, int cap, int32_t *n_out) {
    const int nOct = sp->n_octaves > 0 ? sp->n_octaves : 4, nLay = sp->n_octave_layers > 0 ? sp->n_octave_layers : 2;
    if (nOct > 8 || nLay > 8) return fail(c, FE_ERR_BAD_ARG, "fe_surf_detect: at most 8 octaves / 8 layers");
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    int r = set_geom(c, w, h, n_images);
    if (r != FE_OK) return r;
    if ((r = ensure(c, GRP_FLOAT | GRP_INTEGRAL | GRP_SURFDET)) != FE_OK) return r;
    const Geom &g = c->g;
    Buffers &b = c->b;
    const size_t MI = c->cfg.max_images;
    { StageTimer t(c, ST_H2D); if ((r = upload_images(c, imgs, n_images, stride, 0, 1)) != FE_OK) return r; t.done(0); }
    if ((r = hessian_detect(c, g, b, sp, c->stream, true, nullptr)) != FE_OK) return r;
    // std::sort(keypoints, KeypointGreater()) -- src/surf.cpp:445-460,511 -- as a rank sort on the device
    { StageTimer t(c, ST_SELECT); t.done(launch_surf_rank_sort(b.hes_kp, b.kp, b.hes_count, g.kp_cap, b.hes_count + MI, n_images, c->stream)); }
    FE_CUDA(c, cudaGetLastError());
    std::vector<uint32_t> hc(2 * MI);
    FE_CUDA(c, cudaMemcpyAsync(hc.data(), b.hes_count, sizeof(uint32_t) * 2 * MI, cudaMemcpyDeviceToHost, c->stream));
    FE_CUDA(c, cudaStreamSynchronize(c->stream));
    int max_win = 0;
    bool over = false;
    for (int i = 0; i < n_images; ++i) {
        if ((int)hc[i] > g.kp_cap) { over = true; n_out[i] = (int32_t)hc[i]; }
        float ms;
        memcpy(&ms, &hc[MI + i], 4);
        max_win = std::max(max_win, (int)(21.f * (ms * 1.2f / 9.0f)));
    }
    if (over) return fail(c, FE_ERR_CAPACITY, "fe_surf_detect: more keypoints than fe_config.max_keypoints");
    // orientation + descriptors for every keypoint (SURFInvoker runs even when no descriptors are requested: it assigns the
    // orientation and marks keypoints for deletion, src/surf.cpp:940-978)
    const bool upright = sp->upright != 0, ext = sp->extended != 0;
    const int dim = ext ? 128 : 64;
    { StageTimer t(c, ST_SURF); t.done(launch_surf(g, b, b.hes_count, ext, upright, std::max(max_win, 1), c->stream)); }
    FE_CUDA(c, cudaGetLastError());
    std::vector<fe_kpoint> det;
    std::vector<float> dd;
    bool cap_over = false;
    for (int i = 0; i < n_images; ++i) {
        const int found = (int)hc[i];
        det.resize(std::max(found, 1));
        if (found > 0) {
            FE_CUDA(c, cudaMemcpyAsync(det.data(), b.kp + (size_t)i * g.kp_cap, sizeof(fe_kpoint) * found, cudaMemcpyDeviceToHost, c->stream));
            if (desc) {
                dd.resize((size_t)found * dim);
                FE_CUDA(c, cudaMemcpy2DAsync(dd.data(), sizeof(float) * dim, b.fdesc + (size_t)i * g.kp_cap * 128, sizeof(float) * 128,
                                             sizeof(float) * dim, found, cudaMemcpyDeviceToHost, c->stream));
            }
            FE_CUDA(c, cudaStreamSynchronize(c->stream));
        }
        int m = 0;
        fe_kpoint *ko = kps + (size_t)i * cap;
        float *dout = desc ? desc + (size_t)i * cap * dim : nullptr;
        for (int k = 0; k < found; ++k) {
            if (!(det[k].size > 0)) continue;          // marked for deletion
            if (m < cap) {
                ko[m] = det[k];
                if (dout) memcpy(dout + (size_t)m * dim, dd.data() + (size_t)k * dim, sizeof(float) * dim);
            }
            ++m;
        }
        n_out[i] = m;
        cap_over |= m > cap;
    }
    if ((r = sync_and_resolve(c)) != FE_OK) return r;
    if (cap_over) return fail(c, FE_ERR_CAPACITY, "fe_surf_detect: more keypoints than capacity");
    return FE_OK;
}

int32_t fe_surf_detect_and_compute(fe_ctx *c, const uint8_t *img, int32_t w, int32_t h, int32_t stride,
                                   const fe_surf_params *sp, fe_kpoint *kps, float *desc, int32_t cap, int32_t *n) {
    if (!c || !img || !sp || !kps || !n || cap < 1 || stride < w) return fail(c, FE_ERR_BAD_ARG, "fe_surf_detect_and_compute: bad argument");
    return surf_detect_impl(c, 1, img, w, h, stride, sp, kps, desc, cap, n);
}

// The same for a batch of n_images dense images (stride = width): kps [n_images][cap], desc [n_images][cap][64 / 128], n [n_images]
int32_t fe_surf_detect_batch(fe_ctx *c, int32_t n_images, const uint8_t *imgs, int32_t w, int32_t h, const fe_surf_params *sp,
                             fe_kpoint *kps, float *desc, int32_t cap, int32_t *n) {
    if (!c || !imgs || !sp || !kps || !n || cap < 1 || n_images < 1) return fail(c, FE_ERR_BAD_ARG, "fe_surf_detect_batch: bad argument");
    return surf_detect_impl(c, n_images, imgs, w, h, w, sp, kps, desc, cap, n);
}

// upload externally supplied keypoints (+ optional descriptors) into image slot `slot`
static int upload_kps(fe_ctx *c, int slot, const fe_kpoint *kps, const void *desc, int n, int dim = 0, int bin_bytes = 32) {
    const size_t C = c->g.kp_cap;
    if (n > (int)C) return fail(c, FE_ERR_CAPACITY, "more keypoints than fe_config.max_keypoints");
    if (n > 0) {
        FE_CUDA(c, cudaMemcpyAsync(c->b.kp + slot * C, kps, sizeof(fe_kpoint) * n, cudaMemcpyHostToDevice, c->stream));
        if (desc && dim == 0 && bin_bytes == 32)
            FE_CUDA(c, cudaMemcpyAsync(c->b.desc + slot * C * 32, desc, (size_t)32 * n, cudaMemcpyHostToDevice, c->stream));
        if (desc && dim == 0 && bin_bytes < 32) {
            // narrower binary rows (BRIEF-16) ride in the 256-bit rows the matchers read, zero-padded: Hamming distances
            // are unchanged
            FE_CUDA(c, cudaMemsetAsync(c->b.desc + slot * C * 32, 0, (size_t)32 * n, c->stream));
            FE_CUDA(c, cudaMemcpy2DAsync(c->b.desc + slot * C * 32, 32, desc, (size_t)bin_bytes, (size_t)bin_bytes, n,
                                         cudaMemcpyHostToDevice, c->stream));
        }
        if (desc && dim > 0)   // float rows of `dim` -> device rows of 128 floats
            FE_CUDA(c, cudaMemcpy2DAsync(c->b.fdesc + slot * C * 128, sizeof(float) * 128, desc, sizeof(float) * dim,
                                         sizeof(float) * dim, n, cudaMemcpyHostToDevice, c->stream));
    }
    return FE_OK;
}

int32_t fe_describe(fe_ctx *c, const uint8_t *img, int32_t w, int32_t h, int32_t stride, fe_kpoint *kps,
                    int32_t *n_inout, void *desc, int32_t desc_kind) {
    if (!c || !img || !kps || !n_inout || !desc || stride < w || *n_inout < 0) return fail(c, FE_ERR_BAD_ARG, "fe_describe: bad argument");
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    int r = set_geom(c, w, h, 1);
    if (r != FE_OK) return r;
    if (desc_kind == FE_DESC_SURF64 || desc_kind == FE_DESC_SURF128) {
        // cv::SURF::operator()(img, mask, kps, desc, useProvidedKeypoints = true), src/surf.cpp:896-980
        const int n = *n_inout, dim = desc_dim(desc_kind);
        if (n == 0) return FE_OK;
        if (n > c->g.kp_cap) return fail(c, FE_ERR_CAPACITY, "more keypoints than fe_config.max_keypoints");
        int max_win = 0;
        for (int i = 0; i < n; ++i) {
            const int wsz = (int)(21.f * (kps[i].size * 1.2f / 9.0f));
            if (wsz > SURF_DIRECT_MAX_WIN) return fail(c, FE_ERR_UNSUPPORTED, "fe_describe: SURF window above 1024 px (keypoint size > 365) is not supported");
            max_win = std::max(max_win, wsz);
        }
        const bool upright = c->cfg.surf_upright != 0;
        if ((r = ensure(c, GRP_FLOAT | (upright ? 0u : GRP_INTEGRAL))) != FE_OK) return r;
        { StageTimer t(c, ST_H2D);
          if ((r = upload_images(c, img, 1, stride, 0, 1)) != FE_OK) return r;
          if ((r = upload_kps(c, 0, kps, nullptr, n)) != FE_OK) return r;
          c->h_counts[0] = (uint32_t)n;
          FE_CUDA(c, cudaMemcpyAsync(c->b.n_override, c->h_counts, sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
          t.done(0); }
        { StageTimer t(c, ST_SURF); t.done(launch_surf(c->g, c->b, c->b.n_override, dim == 128, upright, max_win, c->stream)); }
        FE_CUDA(c, cudaGetLastError());
        FE_CUDA(c, cudaMemcpyAsync(kps, c->b.kp, sizeof(fe_kpoint) * n, cudaMemcpyDeviceToHost, c->stream));
        FE_CUDA(c, cudaMemcpy2DAsync(desc, sizeof(float) * dim, c->b.fdesc, sizeof(float) * 128, sizeof(float) * dim, n,
                                     cudaMemcpyDeviceToHost, c->stream));
        if ((r = sync_and_resolve(c)) != FE_OK) return r;
        // remove keypoints that were marked for deletion (src/surf.cpp:953-978)
        float *d = static_cast<float *>(desc);
        int m = 0;
        for (int i = 0; i < n; ++i) {
            if (kps[i].size > 0) {
                if (i > m) { kps[m] = kps[i]; memmove(d + (size_t)m * dim, d + (size_t)i * dim, sizeof(float) * dim); }
                ++m;
            }
        }
        *n_inout = m;
        return FE_OK;
    }
    if (brief_width(desc_kind) > 0) {
        // cv::BriefDescriptorExtractor::compute: runByImageBorder(PATCH_SIZE / 2 + KERNEL_SIZE / 2 = 28), integral, tests
        const int bw = brief_width(desc_kind), slot = brief_slot(desc_kind);
        if (!c->brief_bytes[slot]) return fail(c, FE_ERR_UNSUPPORTED, "fe_describe: no BRIEF test table for this width (fe_set_brief_pattern)");
        const int edge = 28;
        int m = 0;
        for (int i = 0; i < *n_inout; ++i) {
            const fe_kpoint &k = kps[i];
            if (k.x >= edge && k.x < w - edge && k.y >= edge && k.y < h - edge) kps[m++] = k;
        }
        *n_inout = m;
        if (m == 0) return FE_OK;
        if (m > c->g.kp_cap) return fail(c, FE_ERR_CAPACITY, "more keypoints than fe_config.max_keypoints");
        if ((r = ensure(c, GRP_INTEGRAL | GRP_BRIEF)) != FE_OK) return r;
        Buffers &bb = c->b;
        { StageTimer t(c, ST_H2D);
          if ((r = upload_images(c, img, 1, stride, 0, 1)) != FE_OK) return r;
          if ((r = upload_kps(c, 0, kps, nullptr, m)) != FE_OK) return r;
          c->h_counts[0] = (uint32_t)m;
          FE_CUDA(c, cudaMemcpyAsync(bb.n_override, c->h_counts, sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
          t.done(0); }
        { StageTimer t(c, ST_BLUR); t.done(launch_integral(c->g, bb, c->stream)); }
        { StageTimer t(c, ST_BRIEF);
          t.done(launch_brief_ext(c->g, bb, bb.n_override, bb.brief_tab + (size_t)slot * 512 * 4, bw, c->brief_orient[slot], bb.brief_desc, 64, c->stream)); }
        FE_CUDA(c, cudaGetLastError());
        FE_CUDA(c, cudaMemcpy2DAsync(desc, (size_t)bw, bb.brief_desc, 64, (size_t)bw, m, cudaMemcpyDeviceToHost, c->stream));
        return sync_and_resolve(c);
    }
    if (desc_kind == FE_DESC_FREAK) {
        // cv::FREAK::computeImpl: scale index per keypoint, erase what does not fit, orientation, 512 pair tests
        if (!c->b.freak_tab) return fail(c, FE_ERR_UNSUPPORTED, "fe_describe: FREAK is not configured (fe_set_freak)");
        const float size_cst = static_cast<float>(64 / (0.693147180559945 * c->freak_octaves));
        std::vector<int32_t> sidx;
        int m = 0;
        for (int i = 0; i < *n_inout; ++i) {
            const fe_kpoint &k = kps[i];
            int si = c->freak_scale_norm ? std::max((int)(std::log((double)(k.size / 7.f)) * size_cst + 0.5), 0)
                                         : std::max((int)(1.0986122886681 * size_cst + 0.5), 0);
            if (si >= 64) si = 63;
            const int ps = c->freak_sizes[si];
            if (k.x <= (float)ps || k.y <= (float)ps || k.x >= (float)(w - ps) || k.y >= (float)(h - ps)) continue;
            kps[m++] = k;
            sidx.push_back(si);
        }
        *n_inout = m;
        if (m == 0) return FE_OK;
        if (m > c->g.kp_cap) return fail(c, FE_ERR_CAPACITY, "more keypoints than fe_config.max_keypoints");
        if ((r = ensure(c, GRP_INTEGRAL | GRP_BRIEF)) != FE_OK) return r;
        Buffers &bb = c->b;
        { StageTimer t(c, ST_H2D);
          if ((r = upload_images(c, img, 1, stride, 0, 1)) != FE_OK) return r;
          if ((r = upload_kps(c, 0, kps, nullptr, m)) != FE_OK) return r;
          c->h_counts[0] = (uint32_t)m;
          FE_CUDA(c, cudaMemcpyAsync(bb.n_override, c->h_counts, sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
          FE_CUDA(c, cudaMemcpyAsync(bb.freak_scale, sidx.data(), sizeof(int32_t) * m, cudaMemcpyHostToDevice, c->stream));
          t.done(0); }
        { StageTimer t(c, ST_BLUR); t.done(launch_integral(c->g, bb, c->stream)); }
        { StageTimer t(c, ST_BRIEF);
          t.done(launch_freak(c->g, bb, bb.n_override, bb.freak_scale, bb.freak_tab, bb.freak_opairs, bb.freak_dpairs, c->freak_orient,
                              bb.brief_desc, c->stream)); }
        FE_CUDA(c, cudaGetLastError());
        FE_CUDA(c, cudaMemcpyAsync(kps, bb.kp, sizeof(fe_kpoint) * m, cudaMemcpyDeviceToHost, c->stream));
        FE_CUDA(c, cudaMemcpyAsync(desc, bb.brief_desc, (size_t)64 * m, cudaMemcpyDeviceToHost, c->stream));
        return sync_and_resolve(c);    // sidx stays alive until here: the copies are complete after the synchronisation
    }
    if (desc_kind != FE_DESC_ORB256) return fail(c, FE_ERR_UNSUPPORTED, "fe_describe: unknown descriptor kind");
    // KeyPointsFilter::runByImageBorder(keypoints, image.size(), edgeThreshold) as ORB.compute does
    const int edge = c->cfg.edge_threshold;       // KeyPointsFilter::runByImageBorder(edgeThreshold), exactly
    int m = 0;
    for (int i = 0; i < *n_inout; ++i) {
        const fe_kpoint &k = kps[i];
        if (k.x >= edge && k.x < w - edge && k.y >= edge && k.y < h - edge) kps[m++] = k;
    }
    *n_inout = m;
    if (m == 0) return FE_OK;
    { StageTimer t(c, ST_H2D);
      if ((r = upload_images(c, img, 1, stride, 0, 1)) != FE_OK) return r;
      if ((r = upload_kps(c, 0, kps, nullptr, m)) != FE_OK) return r;
      c->h_counts[0] = (uint32_t)m;
      FE_CUDA(c, cudaMemcpyAsync(c->b.n_override, c->h_counts, sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
      t.done(0); }
    { StageTimer t(c, ST_ORIENT); t.done(launch_unpack_kps(c->g, c->b, c->b.n_override, c->stream)); }
    { StageTimer t(c, ST_BLUR); t.done(launch_blur(c->g, c->b, c->stream)); }
    { StageTimer t(c, ST_BRIEF); t.done(launch_rbrief(c->g, detect_params(c), c->b, c->b.n_override, c->stream)); }
    FE_CUDA(c, cudaGetLastError());
    FE_CUDA(c, cudaMemcpyAsync(desc, c->b.desc, (size_t)32 * m, cudaMemcpyDeviceToHost, c->stream));
    return sync_and_resolve(c);
}

// shared body of fe_knn2 / fe_stereo_match / fe_window_match: slot 0 = query, slot 1 = train
static int match_host_inputs(fe_ctx *c, const fe_kpoint *qk, const void *qd, int nq, const fe_kpoint *tk,
                             const void *td, int nt, int desc_kind, const fe_match_cfg *cfg) {
    if (!c || !cfg || nq < 0 || nt < 0 || (nq > 0 && (!qk || !qd)) || (nt > 0 && (!tk || !td)))
        return fail(c, FE_ERR_BAD_ARG, "match: bad argument");
    const int dim = desc_dim(desc_kind);
    if ((dim == 0) != (cfg->norm == FE_NORM_HAMMING || cfg->norm == FE_NORM_HAMMING2) || (dim > 0 && cfg->norm != FE_NORM_L2))
        return fail(c, FE_ERR_UNSUPPORTED, "match: ORB256 / BRIEF go with FE_NORM_HAMMING / FE_NORM_HAMMING2, SURF64/128 with FE_NORM_L2");
    const bool wide = desc_kind == FE_DESC_BRIEF64 || desc_kind == FE_DESC_FREAK;      // 512-bit rows (match512.cu)
    if (wide && cfg->norm != FE_NORM_HAMMING) return fail(c, FE_ERR_UNSUPPORTED, "match: BRIEF-64 / FREAK rows go with FE_NORM_HAMMING");
    const int bin_bytes = binary_bytes(desc_kind);
    const bool cross = cfg->mode == FE_MATCH_CROSSCHECK;
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    { int r0 = ensure(c, wide ? GRP_BRIEF : match_groups(dim, cross)); if (r0 != FE_OK) return r0; }
    if (c->cfg.max_images < 2) return fail(c, FE_ERR_CAPACITY, "matching needs fe_config.max_images >= 2");
    // geometry only matters for kp_cap here; keep whatever image geometry is resident
    if (c->g.kp_cap == 0) { int r = set_geom(c, 16, 16, 2); if (r != FE_OK) return r; }
    c->g.n_images = std::max(c->g.n_images, 2);
    int r;
    StageTimer t(c, ST_H2D);
    if ((r = upload_kps(c, 0, qk, wide ? nullptr : qd, nq, dim, bin_bytes)) != FE_OK) return r;
    if ((r = upload_kps(c, 1, tk, wide ? nullptr : td, nt, dim, bin_bytes)) != FE_OK) return r;
    if (wide) {
        const size_t C = c->g.kp_cap;
        if (nq > 0) FE_CUDA(c, cudaMemcpyAsync(c->b.brief_desc, qd, (size_t)64 * nq, cudaMemcpyHostToDevice, c->stream));
        if (nt > 0) FE_CUDA(c, cudaMemcpyAsync(c->b.brief_desc + C * 64, td, (size_t)64 * nt, cudaMemcpyHostToDevice, c->stream));
    }
    c->h_counts[0] = (uint32_t)nq; c->h_counts[1] = (uint32_t)nt;
    FE_CUDA(c, cudaMemcpyAsync(c->b.n_override, c->h_counts, 2 * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
    t.done(0);
    { StageTimer t2(c, ST_ORIENT); t2.done(launch_unpack_kps(c->g, c->b, c->b.n_override, c->stream)); }
    if (wide) {
        if (cross) {
            { StageTimer t2(c, ST_MATCH); t2.done(launch_hamming512_cross(c->g, 1, c->b.brief_desc, c->b, c->b.n_override, c->stream)); }
            { StageTimer t2(c, ST_FINALIZE); t2.done(launch_finalize_cross(c->g, 1, cfg->max_dy, c->b, c->b.n_override, c->stream)); }
        } else {
            { StageTimer t2(c, ST_KNN); t2.done(launch_hamming512_knn2(c->g, 1, match_params(cfg), c->b.brief_desc, c->b, c->b.n_override, c->stream)); }
            { StageTimer t2(c, ST_FINALIZE); t2.done(launch_finalize_ratio(c->g, 1, cfg->ratio, c->b, c->b.n_override, c->stream)); }
        }
        FE_CUDA(c, cudaGetLastError());
        return FE_OK;
    }
    bool sorted = true;
    for (int i = 1; i < nt && sorted; ++i) sorted = !(tk[i].y < tk[i - 1].y);
    if (dim > 0) return run_match_l2_on(c, c->g, c->b, c->stream, true, 1, dim, cross ? nullptr : cfg, cross ? cfg : nullptr, c->b.n_override, sorted);
    bool qsorted = sorted;
    for (int i = 1; i < nq && qsorted; ++i) qsorted = !(qk[i].y < qk[i - 1].y);
    return run_match_on(c, c->g, c->b, c->stream, true, 1, cross ? nullptr : cfg, cross ? cfg : nullptr, c->b.n_override, sorted, qsorted,
                        bin_bytes);
}

int32_t fe_knn2(fe_ctx *c, const fe_kpoint *qk, const void *qd, int32_t nq, const fe_kpoint *tk, const void *td,
                int32_t nt, int32_t desc_kind, const fe_match_cfg *cfg, int32_t *idx, float *dist) {
    if (!idx || !dist) return fail(c, FE_ERR_BAD_ARG, "fe_knn2: null output");
    fe_match_cfg a = cfg ? *cfg : fe_match_cfg{};
    a.mode = FE_MATCH_RATIO;
    int r = match_host_inputs(c, qk, qd, nq, tk, td, nt, desc_kind, &a);
    if (r != FE_OK) return r;
    if (desc_dim(desc_kind) > 0) {
        std::vector<unsigned long long> kb64(nq), ks64(nq);
        if (nq > 0) {
            FE_CUDA(c, cudaMemcpyAsync(kb64.data(), c->b.best64, sizeof(unsigned long long) * nq, cudaMemcpyDeviceToHost, c->stream));
            FE_CUDA(c, cudaMemcpyAsync(ks64.data(), c->b.second64, sizeof(unsigned long long) * nq, cudaMemcpyDeviceToHost, c->stream));
        }
        if ((r = sync_and_resolve(c)) != FE_OK) return r;
        for (int i = 0; i < nq; ++i) {
            const unsigned long long k[2] = {kb64[i], ks64[i]};
            for (int j = 0; j < 2; ++j) {
                const bool none = k[j] == ~0ull;
                uint32_t bits = (uint32_t)(k[j] >> 32);
                float d2;
                memcpy(&d2, &bits, 4);
                idx[2 * i + j] = none ? -1 : (int32_t)(k[j] & 0xFFFFFFFFu);
                dist[2 * i + j] = none ? __builtin_inff() : sqrtf(d2);
            }
        }
        return FE_OK;
    }
    std::vector<uint32_t> kb(nq), ks(nq);
    if (nq > 0) {
        FE_CUDA(c, cudaMemcpyAsync(kb.data(), c->b.best, sizeof(uint32_t) * nq, cudaMemcpyDeviceToHost, c->stream));
        FE_CUDA(c, cudaMemcpyAsync(ks.data(), c->b.second, sizeof(uint32_t) * nq, cudaMemcpyDeviceToHost, c->stream));
    }
    if ((r = sync_and_resolve(c)) != FE_OK) return r;
    for (int i = 0; i < nq; ++i) {
        const uint32_t k[2] = {kb[i], ks[i]};
        for (int j = 0; j < 2; ++j) {
            idx[2 * i + j] = k[j] == KEY_NONE ? -1 : (int32_t)(k[j] & 0xFFFF);
            dist[2 * i + j] = k[j] == KEY_NONE ? __builtin_inff() : (float)(k[j] >> 16);
        }
    }
    return FE_OK;
}

int32_t fe_stereo_match(fe_ctx *c, const fe_kpoint *lk, const void *ld, int32_t nl, const fe_kpoint *rk,
                        const void *rd, int32_t nr, int32_t desc_kind, const fe_match_cfg *cfg, fe_match *out,
                        int32_t cap, int32_t *n) {
    if (!n || cap < 0 || (cap > 0 && !out)) return fail(c, FE_ERR_BAD_ARG, "fe_stereo_match: bad output");
    int r = match_host_inputs(c, lk, ld, nl, rk, rd, nr, desc_kind, cfg);
    if (r != FE_OK) return r;
    const bool cross = cfg->mode == FE_MATCH_CROSSCHECK;
    FE_CUDA(c, cudaMemcpyAsync(c->h_counts, cross ? c->b.n_b : c->b.n_a, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    FE_CUDA(c, cudaStreamSynchronize(c->stream));
    const int found = (int)c->h_counts[0];
    *n = found;
    const int m = std::min(found, cap);
    if (m > 0) FE_CUDA(c, cudaMemcpyAsync(out, cross ? c->b.match_b : c->b.match_a, sizeof(fe_match) * m, cudaMemcpyDeviceToHost, c->stream));
    if ((r = sync_and_resolve(c)) != FE_OK) return r;
    if (found > cap) return fail(c, FE_ERR_CAPACITY, "fe_stereo_match: more matches than capacity");
    return FE_OK;
}

int32_t fe_window_match(fe_ctx *c, const fe_kpoint *ck, const void *cd, int32_t nc, const fe_kpoint *pk,
                        const void *pd, int32_t np, int32_t desc_kind, const fe_match_cfg *cfg, fe_match *out,
                        int32_t cap, int32_t *n) {
    if (!cfg) return fail(c, FE_ERR_BAD_ARG, "fe_window_match: null cfg");
    fe_match_cfg w = *cfg;
    w.mode = FE_MATCH_RATIO;
    w.mask = FE_MASK_WINDOW;
    if (w.win_w <= 0) w.win_w = 100;
    if (w.win_h <= 0) w.win_h = 100;
    return fe_stereo_match(c, ck, cd, nc, pk, pd, np, desc_kind, &w, out, cap, n);
}

// srv/windowMatching.srv (bool reset, stereoLandmarks latestFrame -> windowStatus state) / WindowMatcher::newStereo's
// window (src/WindowMatcher.cpp:92-102): the previous frame's landmark list stays on the device, every update uploads only
// the new frame, matches it against the previous one and shifts the window.
int32_t fe_window_update(fe_ctx *c, int32_t reset, const fe_kpoint *l_kps, const void *l_desc, const void *r_desc, int32_t n,
                         int32_t desc_kind, const fe_match_cfg *cfg, const fe_window_cfg *wc, fe_match *tracks, int32_t cap,
                         int32_t *n_tracks, int32_t *frames_in_window) {
    if (!c) return FE_ERR_BAD_ARG;
    if (reset) {       // window.update(reset): every list is cleared, an empty response goes back
        c->wu_frames = 0; c->wu_prev_n = 0;
        if (n_tracks) *n_tracks = 0;
        if (frames_in_window) *frames_in_window = 0;
        return FE_OK;
    }
    if (!cfg || !n_tracks || n < 0 || (n > 0 && (!l_kps || !l_desc)) || cap < 0 || (cap > 0 && !tracks))
        return fail(c, FE_ERR_BAD_ARG, "fe_window_update: bad argument");
    const bool live = cfg->mode == FE_MATCH_CROSSCHECK;
    const int dim = desc_dim(desc_kind);      // SURF-64 / SURF-128 float rows; 0 = binary
    if (dim == 0 && desc_kind != FE_DESC_ORB256 && desc_kind != FE_DESC_BRIEF16 && desc_kind != FE_DESC_BRIEF32)
        return fail(c, FE_ERR_UNSUPPORTED, "fe_window_update: binary descriptors of up to 256 bits, or SURF-64 / SURF-128");
    if (dim == 0 && cfg->norm != FE_NORM_HAMMING && cfg->norm != FE_NORM_HAMMING2) return fail(c, FE_ERR_UNSUPPORTED, "fe_window_update: Hamming norms");
    if (dim > 0 && cfg->norm != FE_NORM_L2) return fail(c, FE_ERR_UNSUPPORTED, "fe_window_update: SURF rows are matched with FE_NORM_L2");
    if (live && !r_desc && n > 0) return fail(c, FE_ERR_BAD_ARG, "fe_window_update: the liveGraph variant needs the right descriptors");
    if (live && cfg->mask != FE_MASK_NONE) return fail(c, FE_ERR_BAD_ARG, "fe_window_update: cross-check takes no mask (BFMatcher asserts)");
    if (c->wu_frames >= 1 && dim != c->wu_dim)
        return fail(c, FE_ERR_BAD_ARG, "fe_window_update: the previous frame's rows are of another kind (binary, SURF-64, SURF-128): reset the window first");
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    const size_t C = c->cfg.max_keypoints;
    if (n > (int)C) return fail(c, FE_ERR_CAPACITY, "more landmarks than fe_config.max_keypoints");
    int r;
    if ((r = ensure(c, GRP_WUPDATE | (dim > 0 ? match_groups(dim, false) | GRP_WUFLOAT : live ? GRP_WLIVE : 0u))) != FE_OK) return r;
    Buffers &b = c->b;
    if (c->g.kp_cap == 0 && (r = set_geom(c, 16, 16, 2)) != FE_OK) return r;
    const int bin_bytes = binary_bytes(desc_kind);
    auto put_desc = [&](uint8_t *dst, const void *src) -> int {
        if (bin_bytes == 32) { FE_CUDA(c, cudaMemcpyAsync(dst, src, (size_t)32 * n, cudaMemcpyHostToDevice, c->stream)); }
        else {
            FE_CUDA(c, cudaMemsetAsync(dst, 0, (size_t)32 * n, c->stream));
            FE_CUDA(c, cudaMemcpy2DAsync(dst, 32, src, (size_t)bin_bytes, (size_t)bin_bytes, n, cudaMemcpyHostToDevice, c->stream));
        }
        return FE_OK;
    };
    // float rows of dim floats -> device rows of 128 floats (fdesc's stride, which the L2 matchers read)
    auto put_rows = [&](float *dst, const void *src) -> int {
        FE_CUDA(c, cudaMemcpy2DAsync(dst, sizeof(float) * 128, src, sizeof(float) * dim, sizeof(float) * dim, n, cudaMemcpyHostToDevice,
                                     c->stream));
        return FE_OK;
    };
    {   // slot 0 <- the new frame
        StageTimer t(c, ST_H2D);
        if (n > 0) {
            FE_CUDA(c, cudaMemcpyAsync(b.wu_kp, l_kps, sizeof(fe_kpoint) * n, cudaMemcpyHostToDevice, c->stream));
            if (dim > 0) {
                if ((r = put_rows(b.wu_fdesc, l_desc)) != FE_OK) return r;
                if (r_desc && (r = put_rows(b.wu_frdesc, r_desc)) != FE_OK) return r;
            } else {
                if ((r = put_desc(b.wu_desc, l_desc)) != FE_OK) return r;
                if (r_desc && (r = put_desc(b.wu_rdesc, r_desc)) != FE_OK) return r;
            }
        }
        c->h_counts[0] = (uint32_t)n; c->h_counts[1] = (uint32_t)c->wu_prev_n;
        FE_CUDA(c, cudaMemcpyAsync(b.wu_n, c->h_counts, 2 * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
        t.done(0);
    }
    Geom gv = c->g;
    gv.n_images = 2;
    Buffers v = b;
    v.kp = b.wu_kp; v.kx = b.wu_kx; v.ky = b.wu_ky; v.kcs = b.wu_kcs; v.desc = b.wu_desc; v.fdesc = b.wu_fdesc;
    { StageTimer t(c, ST_ORIENT); t.done(launch_unpack_kps(gv, v, b.wu_n, c->stream)); }   // (re-derives the previous frame's kx / ky too)
    bool sorted = true;        // raster order of the new frame's landmarks: the banded kernel's precondition when it is the train side next time
    for (int i = 1; i < n && sorted; ++i) sorted = !(l_kps[i].y < l_kps[i - 1].y);
    // window.push_back(current); if (window.size() >= nWindow) erase(begin)   [C++ node: at most nWindow - 1 frames stay]
    // window.append(frame); if len >= length + 1: del window[0]               [Python service: `length` frames stay]
    const bool py = wc && wc->variant == 1;
    const int len = wc && wc->length > 0 ? wc->length : (py ? 2 : 3);     // window(length = 2) / WindowMatcher slidingWindow(3)
    int frames = c->wu_frames + 1;
    if (py) { if (frames >= len + 1) frames = len; }
    else if (frames >= len) frames = std::max(len - 1, 0);
    int found = 0;
    if (c->wu_frames >= 1 && frames > 1) {      // window.size() > 1: match against window[size - 2]
        if (live && dim > 0) {
            // liveGraph applies no |dy| filter: the exact all-pairs FP32 pass on the left and on the right rows.  The right
            // side's keys use the ratio-mode key arrays, which cross-check mode leaves free.
            Buffers vl = v, vr = v;
            vr.fdesc = b.wu_frdesc; vr.allbest64 = b.best64; vr.colbest64 = b.second64;
            const MatchParams none = match_params(nullptr);
            { StageTimer t(c, ST_L2);
              t.done(launch_l2_match(gv, 1, dim, none, false, true, vl, b.wu_n, c->stream) +
                     launch_l2_match(gv, 1, dim, none, false, true, vr, b.wu_n, c->stream)); }
            { StageTimer t(c, ST_FINALIZE);
              t.done(launch_l2_finalize_cross_both(gv, 1, b.wu_n, b.allbest64, b.colbest64, b.best64, b.second64, b.match_b, b.n_b,
                                                   c->stream)); }
            FE_CUDA(c, cudaGetLastError());
        } else if (live) {
            const bool h2 = cfg->norm == FE_NORM_HAMMING2;
            Buffers vl = v, vr = v;
            vl.allbest = b.allbest; vl.colbest = b.colbest;
            vr.desc = b.wu_rdesc; vr.allbest = b.wbest_r; vr.colbest = b.wcol_r;
            { StageTimer t(c, ST_MATCH);
              t.done(launch_hamming_cross(gv, 1, h2, vl, b.wu_n, c->stream) + launch_hamming_cross(gv, 1, h2, vr, b.wu_n, c->stream)); }
            { StageTimer t(c, ST_FINALIZE);
              t.done(launch_finalize_cross_both(gv, 1, b.wu_n, b.allbest, b.colbest, b.wbest_r, b.wcol_r, b.match_b, b.n_b, c->stream)); }
            FE_CUDA(c, cudaGetLastError());
        } else {
            fe_match_cfg w = *cfg;
            w.mode = FE_MATCH_RATIO;
            if (w.mask == FE_MASK_WINDOW) { if (w.win_w <= 0) w.win_w = 100; if (w.win_h <= 0) w.win_h = 100; }
            if (dim > 0) r = run_match_l2_on(c, gv, v, c->stream, true, 1, dim, &w, nullptr, b.wu_n, c->wu_prev_sorted);
            else r = run_match_on(c, gv, v, c->stream, true, 1, &w, nullptr, b.wu_n, c->wu_prev_sorted, false, bin_bytes);
            if (r != FE_OK) return r;
        }
        FE_CUDA(c, cudaMemcpyAsync(c->h_counts, live ? b.n_b : b.n_a, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
        FE_CUDA(c, cudaStreamSynchronize(c->stream));
        found = (int)c->h_counts[0];
        const int m = std::min(found, cap);
        if (m > 0) FE_CUDA(c, cudaMemcpyAsync(tracks, live ? b.match_b : b.match_a, sizeof(fe_match) * m, cudaMemcpyDeviceToHost, c->stream));
    }
    // shift: the new frame becomes the previous one (device-to-device, ~70 bytes per binary landmark, 4 * dim + 28 per SURF one)
    if (n > 0) {
        FE_CUDA(c, cudaMemcpyAsync(b.wu_kp + C, b.wu_kp, sizeof(fe_kpoint) * n, cudaMemcpyDeviceToDevice, c->stream));
        if (dim > 0) {
            const size_t pitch = sizeof(float) * 128;
            FE_CUDA(c, cudaMemcpy2DAsync(b.wu_fdesc + C * 128, pitch, b.wu_fdesc, pitch, sizeof(float) * dim, n, cudaMemcpyDeviceToDevice, c->stream));
            if (r_desc)
                FE_CUDA(c, cudaMemcpy2DAsync(b.wu_frdesc + C * 128, pitch, b.wu_frdesc, pitch, sizeof(float) * dim, n, cudaMemcpyDeviceToDevice,
                                             c->stream));
        } else {
            FE_CUDA(c, cudaMemcpyAsync(b.wu_desc + C * 32, b.wu_desc, (size_t)32 * n, cudaMemcpyDeviceToDevice, c->stream));
            if (r_desc) FE_CUDA(c, cudaMemcpyAsync(b.wu_rdesc + C * 32, b.wu_rdesc, (size_t)32 * n, cudaMemcpyDeviceToDevice, c->stream));
        }
    }
    c->wu_prev_n = n; c->wu_prev_sorted = sorted; c->wu_frames = frames; c->wu_dim = dim;
    *n_tracks = found;
    if (frames_in_window) *frames_in_window = frames;
    if ((r = sync_and_resolve(c)) != FE_OK) return r;
    if (found > cap) return fail(c, FE_ERR_CAPACITY, "fe_window_update: more tracks than capacity");
    return FE_OK;
}

// ---- batched pipeline ------------------------------------------------------------------------------

int32_t fe_batch_upload(fe_ctx *c, int32_t n_pairs, const uint8_t *left, const uint8_t *right, int32_t w, int32_t h) {
    if (!c || !left || !right || n_pairs < 1) return fail(c, FE_ERR_BAD_ARG, "fe_batch_upload: bad argument");
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    int r = set_geom(c, w, h, 2 * n_pairs);
    if (r != FE_OK) return r;
    StageTimer t(c, ST_H2D);
    if ((r = upload_images(c, left, n_pairs, w, 0, 2)) != FE_OK) return r;
    if ((r = upload_images(c, right, n_pairs, w, 1, 2)) != FE_OK) return r;
    t.done(0);
    c->h2d_bytes += (int64_t)2 * n_pairs * w * h;
    return FE_OK;
}

// fe_window_batch on a SURF batch: the landmarks' float rows gathered into virtual pairs (g: the resident batch, gv: its
// 2 (F - 1) virtual-pair slots) and matched by the L2 kernels.
static int window_batch_l2(fe_ctx *c, const Geom &g, const Geom &gv, const fe_match_cfg *cfg, bool live, int dim) {
    const int F = g.n_images / 2, V = F - 1;
    Buffers &b = c->b;
    { StageTimer t(c, ST_ORIENT); t.done(launch_gather_landmarks(g, F, b, 0, dim, b.wfdesc, b.wkx, b.wky, b.wcount, c->stream)); }
    Buffers v = b;
    v.fdesc = b.wfdesc; v.kx = b.wkx; v.ky = b.wky;
    v.best64 = b.wbest64; v.second64 = b.wsecond64; v.match_a = b.wmatch; v.n_a = b.wn;
    if (live) {
        // liveGraph applies no |dy| filter, so there are no band candidates for the tensor-core cross-check: the exact
        // all-pairs FP32 pass on the left rows and on the right rows, then the same-landmark intersection
        { StageTimer t(c, ST_ORIENT); t.done(launch_gather_landmarks(g, F, b, 1, dim, b.wfdesc_r, nullptr, nullptr, b.wcount, c->stream)); }
        Buffers vl = v, vr = v;
        vl.allbest64 = b.wbest64; vl.colbest64 = b.wsecond64;
        vr.fdesc = b.wfdesc_r; vr.allbest64 = b.wbest64_r; vr.colbest64 = b.wcol64_r;
        const MatchParams none = match_params(nullptr);
        { StageTimer t(c, ST_L2);
          t.done(launch_l2_match(gv, V, dim, none, false, true, vl, b.wcount, c->stream) +
                 launch_l2_match(gv, V, dim, none, false, true, vr, b.wcount, c->stream)); }
        { StageTimer t(c, ST_FINALIZE);
          t.done(launch_l2_finalize_cross_both(gv, V, b.wcount, b.wbest64, b.wsecond64, b.wbest64_r, b.wcol64_r, b.wmatch, b.wn,
                                               c->stream)); }
        FE_CUDA(c, cudaGetLastError());
        return FE_OK;
    }
    // landmarks inherit the left keypoints' order
    return run_match_l2_on(c, gv, v, c->stream, true, V, dim, cfg, nullptr, b.wcount, batch_raster(c));
}

// WindowMatcher::newStereo matching stage for a whole resident sequence (src/WindowMatcher.cpp:75-231).
int32_t fe_window_batch(fe_ctx *c, const fe_match_cfg *cfg, const double *Q, int32_t cap, fe_match *tracks,
                        int32_t *n_tracks, double *xyz) {
    if (!c || !cfg || cap < 0 || (cap > 0 && !tracks) || !n_tracks) return fail(c, FE_ERR_BAD_ARG, "fe_window_batch: bad argument");
    if (c->g.n_images < 4) return fail(c, FE_ERR_BAD_ARG, "fe_window_batch: run fe_batch_run on at least two frames first");
    const int rows = batch_rows(c), dim = desc_dim(rows);     // SURF-64 / SURF-128 batches: float rows and FE_NORM_L2
    const bool hamming = cfg->norm == FE_NORM_HAMMING || cfg->norm == FE_NORM_HAMMING2;
    if (dim == 0 && !hamming)
        return fail(c, FE_ERR_UNSUPPORTED, "fe_window_batch: ORB-256 / BRIEF sequences are matched with FE_NORM_HAMMING / FE_NORM_HAMMING2");
    if (dim > 0 && cfg->norm != FE_NORM_L2) return fail(c, FE_ERR_UNSUPPORTED, "fe_window_batch: SURF sequences are matched with FE_NORM_L2");
    const bool live = cfg->mode == FE_MATCH_CROSSCHECK;       // liveGraph variant (algorithm.py:1160-1190)
    if (!live && (cfg->mode != FE_MATCH_RATIO || cfg->mask != FE_MASK_WINDOW))
        return fail(c, FE_ERR_BAD_ARG, "fe_window_batch: cfg must be ratio mode with the window mask, or cross-check mode (liveGraph)");
    if (live && cfg->mask != FE_MASK_NONE) return fail(c, FE_ERR_BAD_ARG, "fe_window_batch: cross-check takes no mask (BFMatcher asserts)");
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    const Geom &g = c->g;
    const int F = g.n_images / 2, V = F - 1;
    int r = ensure(c, GRP_WINDOW | (dim > 0 ? match_groups(dim, false) | GRP_WFLOAT | (live ? GRP_WFLIVE : 0u) : live ? GRP_WLIVE : 0u));
    if (r != FE_OK) return r;
    Buffers &b = c->b;
    Geom gv = g;
    gv.n_images = 2 * V;
    if (dim > 0) r = window_batch_l2(c, g, gv, cfg, live, dim);
    else {
        { StageTimer t(c, ST_ORIENT); t.done(launch_gather_landmarks(g, F, b, 0, b.wdesc, b.wkx, b.wky, b.wcount, c->stream)); }
        // the stereo matcher's kernels on the virtual pairs: a Buffers view whose inputs / outputs are the w* arrays
        Buffers v = b;
        v.desc = b.wdesc; v.kx = b.wkx; v.ky = b.wky;
        v.best = b.wbest; v.second = b.wsecond; v.match_a = b.wmatch; v.n_a = b.wn;
        if (live) {
            // cur <-> prev cross-check on the LEFT descriptors and on the RIGHT descriptors, then the same-landmark intersection
            { StageTimer t(c, ST_ORIENT); t.done(launch_gather_landmarks(g, F, b, 1, b.wdesc_r, nullptr, nullptr, b.wcount, c->stream)); }
            const bool h2 = cfg->norm == FE_NORM_HAMMING2;
            Buffers vl = b, vr = b;
            vl.desc = b.wdesc; vl.allbest = b.wbest; vl.colbest = b.wsecond;
            vr.desc = b.wdesc_r; vr.allbest = b.wbest_r; vr.colbest = b.wcol_r;
            { StageTimer t(c, ST_MATCH);
              t.done(launch_hamming_cross(gv, V, h2, vl, b.wcount, c->stream) + launch_hamming_cross(gv, V, h2, vr, b.wcount, c->stream)); }
            { StageTimer t(c, ST_FINALIZE);
              t.done(launch_finalize_cross_both(gv, V, b.wcount, b.wbest, b.wsecond, b.wbest_r, b.wcol_r, b.wmatch, b.wn, c->stream)); }
            FE_CUDA(c, cudaGetLastError());
        } else {
            // landmarks inherit the left keypoints' order
            r = run_match_on(c, gv, v, c->stream, true, V, cfg, nullptr, b.wcount, batch_raster(c), false, binary_bytes(rows));
        }
    }
    if (r != FE_OK) return r;
    if (Q && xyz) {
        FE_CUDA(c, cudaMemcpyAsync(b.wq, Q, sizeof(double) * 16, cudaMemcpyHostToDevice, c->stream));
        StageTimer t(c, ST_FINALIZE);
        t.done(launch_triangulate(g, F, b, b.wq, b.wxyz, c->stream));
    }
    FE_CUDA(c, cudaMemcpyAsync(c->h_counts, b.wn, sizeof(uint32_t) * V, cudaMemcpyDeviceToHost, c->stream));
    FE_CUDA(c, cudaMemcpyAsync(c->h_counts + V, b.n_a, sizeof(uint32_t) * F, cudaMemcpyDeviceToHost, c->stream));
    FE_CUDA(c, cudaStreamSynchronize(c->stream));
    bool overflow = false;
    int max_t = 0, max_l = 0;
    for (int i = 0; i < V; ++i) {
        n_tracks[i] = (int32_t)c->h_counts[i];
        if (n_tracks[i] > cap) overflow = true;
        max_t = std::max(max_t, std::min(n_tracks[i], cap));
    }
    for (int i = 0; i < F; ++i) max_l = std::max(max_l, std::min(std::min((int)c->h_counts[V + i], cap), g.kp_cap));
    if (max_t > 0)
        FE_CUDA(c, cudaMemcpy2DAsync(tracks, sizeof(fe_match) * (size_t)cap, b.wmatch, sizeof(fe_match) * (size_t)g.kp_cap,
                                     sizeof(fe_match) * (size_t)max_t, V, cudaMemcpyDeviceToHost, c->stream));
    if (Q && xyz && max_l > 0)
        FE_CUDA(c, cudaMemcpy2DAsync(xyz, sizeof(double) * 3 * (size_t)cap, b.wxyz, sizeof(double) * 3 * (size_t)g.kp_cap,
                                     sizeof(double) * 3 * (size_t)max_l, F, cudaMemcpyDeviceToHost, c->stream));
    if ((r = sync_and_resolve(c)) != FE_OK) return r;
    if (overflow) return fail(c, FE_ERR_CAPACITY, "fe_window_batch: more tracks than capacity");
    return FE_OK;
}

// cv::ORB::setPatchSize (bin/detect_node:50-51: cv2.ORB_create(); setPatchSize(70) as the descriptor of the live
// Python node).  patchSize != 31 makes OpenCV draw the 512 BRIEF points with makeRandomPattern: cv::RNG(0x34985739),
// x then y uniform in [-patchSize/2, patchSize/2] -- a multiply-with-carry generator restated here and pinned against
// cv2 4.13 through the descriptors it produces.
static const int8_t kBitPattern31[1024] = {
#define FE_PAT_FLAT
#include "orb_pattern_flat.inc"
#undef FE_PAT_FLAT
};

struct CvRng {      // cv::RNG: multiply-with-carry
    uint64_t state;
    uint32_t next() { state = (uint64_t)(uint32_t)state * 4164903690ull + (uint32_t)(state >> 32); return (uint32_t)state; }
    int uniform(int a, int b) { return a + (int)(next() % (uint32_t)(b - a)); }
};

// orb.cpp: pattern0 = bit_pattern_31_ (patch 31) or makeRandomPattern(patchSize) (RNG 0x34985739); WTA_K 2 uses it as is,
// WTA_K 3 / 4 draw 128 tuples of distinct points from it (initializeOrbPattern, RNG 0x12345678).
static int upload_orb_pattern(fe_ctx *c, int patch_size, int wta_k) {
    int8_t base[1024];
    if (patch_size == 31) {
        memcpy(base, kBitPattern31, sizeof(base));
    } else {
        CvRng rng{0x34985739ull};
        const int lo = -(patch_size / 2), hi = patch_size / 2 + 1;
        for (int i = 0; i < 1024; ++i) base[i] = (int8_t)rng.uniform(lo, hi);
    }
    int8_t pat[1024] = {0};
    if (wta_k == 2) {
        memcpy(pat, base, sizeof(pat));
    } else {
        CvRng rng{0x12345678ull};
        for (int i = 0; i < 128; ++i)
            for (int k = 0; k < wta_k; ++k)
                for (;;) {
                    const int idx = rng.uniform(0, 512);
                    const int8_t px = base[2 * idx], py = base[2 * idx + 1];
                    int k1 = 0;
                    for (; k1 < k; ++k1)
                        if (pat[2 * (wta_k * i + k1)] == px && pat[2 * (wta_k * i + k1) + 1] == py) break;
                    if (k1 == k) { pat[2 * (wta_k * i + k)] = px; pat[2 * (wta_k * i + k) + 1] = py; break; }
                }
    }
    FE_CUDA(c, cudaMemcpyAsync(c->b.pattern, pat, sizeof(pat), cudaMemcpyHostToDevice, c->stream));
    // umax of the intensity-centroid disc (orb.cpp): radius halfPatchSize = patchSize / 2
    int umax[128] = {0};
    const int half = patch_size / 2;
    const int vmax = (int)std::floor(half * std::sqrt(2.f) / 2 + 1), vmin = (int)std::ceil(half * std::sqrt(2.f) / 2);
    for (int v = 0; v <= vmax; ++v) umax[v] = (int)lrint(std::sqrt((double)half * half - v * v));
    for (int v = half, v0 = 0; v >= vmin; --v) {
        while (umax[v0] == umax[v0 + 1]) ++v0;
        umax[v] = v0;
        ++v0;
    }
    FE_CUDA(c, cudaMemcpyAsync(c->b.umax, umax, sizeof(umax), cudaMemcpyHostToDevice, c->stream));
    FE_CUDA(c, cudaStreamSynchronize(c->stream));
    return FE_OK;
}

int32_t fe_set_orb_patch_size(fe_ctx *c, int32_t patch_size) {
    if (!c) return FE_ERR_BAD_ARG;
    if (patch_size < 2 || patch_size > 250) return fail(c, FE_ERR_BAD_ARG, "fe_set_orb_patch_size: 2 <= patchSize <= 250");
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    int r = upload_orb_pattern(c, patch_size, c->wta_k);
    if (r != FE_OK) return r;
    c->patch_size = patch_size;
    return FE_OK;
}

// cv::ORB WTA_K (ORB_create(..., WTA_K, ...): features.py:378-387 sweeps 2 / 3 / 4; src/StereoCamera.cpp:504-511 switches
// the matcher to NORM_HAMMING2 when WTA_K > 2).
int32_t fe_set_orb_wta_k(fe_ctx *c, int32_t wta_k) {
    if (!c) return FE_ERR_BAD_ARG;
    if (wta_k < 2 || wta_k > 4) return fail(c, FE_ERR_BAD_ARG, "fe_set_orb_wta_k: WTA_K must be 2, 3 or 4");
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    int r = upload_orb_pattern(c, c->patch_size, wta_k);
    if (r != FE_OK) return r;
    c->wta_k = wta_k;
    return FE_OK;
}

// cv::ORB scoreType (the `score` field of front_end/setDetector: src/StereoCamera.cpp:445,462; src/utils.cpp:86-90).
int32_t fe_set_orb_score_type(fe_ctx *c, int32_t score_type) {
    if (!c) return FE_ERR_BAD_ARG;
    if (score_type != 0 && score_type != 1) return fail(c, FE_ERR_BAD_ARG, "fe_set_orb_score_type: 0 = HARRIS_SCORE, 1 = FAST_SCORE");
    if (score_type == 0 && (!c->cfg.orientation || c->cfg.fast_type != FE_FAST_9_16 || !c->cfg.nonmax))
        return fail(c, FE_ERR_UNSUPPORTED, "fe_set_orb_score_type: HARRIS_SCORE is cv::ORB's (FAST-9_16, NMS, orientation)");
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    if (score_type == 0) { const int r = ensure(c, GRP_HARRIS); if (r != FE_OK) return r; }
    c->score_type = score_type;
    return FE_OK;
}

// cv::ORB nlevels / scaleFactor (ORB_create(nfeatures, scaleFactor, nlevels, ...): features.py:378-387, src/utils.cpp:84-94).
int32_t fe_set_orb_pyramid(fe_ctx *c, int32_t nlevels, float scale_factor) {
    if (!c) return FE_ERR_BAD_ARG;
    if (nlevels < 1 || nlevels > 16 || !(scale_factor > 1.f)) return fail(c, FE_ERR_BAD_ARG, "fe_set_orb_pyramid: 1 <= nlevels <= 16, scaleFactor > 1");
    if (nlevels > 1 && (!c->cfg.orientation || c->cfg.fast_type != FE_FAST_9_16 || !c->cfg.nonmax || c->cfg.n_features < 0))   // (any WTA_K, any patch size)
        return fail(c, FE_ERR_UNSUPPORTED, "fe_set_orb_pyramid: the pyramid is ORB's (FAST-9_16, NMS, orientation, n_features >= 0, patch 31)");
    c->nlevels = nlevels;
    c->scale_factor = (double)scale_factor;
    return FE_OK;
}

// stereoLandmarks of every pair of the resident batch (algorithm_one's packing, src/front_end/algorithm.py:893-913).
int32_t fe_batch_landmarks(fe_ctx *c, int32_t which, int32_t cap, fe_kpoint *l_kps, void *l_desc, fe_kpoint *r_kps,
                           void *r_desc, fe_match *matches, int32_t *n) {
    if (!c || !n || cap < 0 || (which != 0 && which != 1)) return fail(c, FE_ERR_BAD_ARG, "fe_batch_landmarks: bad argument");
    if (c->g.n_images < 2) return fail(c, FE_ERR_BAD_ARG, "fe_batch_landmarks: run fe_batch_run first");
    const int rows = batch_rows(c), dim = desc_dim(rows);     // SURF batches: rows of dim floats; binary ones: binary_bytes(rows)
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    const Geom &g = c->g;
    const int P = g.n_images / 2;
    int r = ensure(c, GRP_LANDMARKS | (dim > 0 ? GRP_LMFLOAT : 0u));
    if (r != FE_OK) return r;
    Buffers &b = c->b;
    const uint32_t *cnt = which == 0 ? b.n_a : b.n_b;
    const fe_match *src = which == 0 ? b.match_a : b.match_b;
    { StageTimer t(c, ST_FINALIZE);
      t.done(dim > 0 ? launch_pack_landmarks(g, P, b, cnt, src, b.lm_lkp, b.lm_rkp, dim, b.lm_lfdesc, b.lm_rfdesc, b.lm_match, c->stream)
                     : launch_pack_landmarks(g, P, b, cnt, src, b.lm_lkp, b.lm_rkp, b.lm_ldesc, b.lm_rdesc, b.lm_match, c->stream)); }
    FE_CUDA(c, cudaGetLastError());
    FE_CUDA(c, cudaMemcpyAsync(c->h_counts, cnt, sizeof(uint32_t) * P, cudaMemcpyDeviceToHost, c->stream));
    FE_CUDA(c, cudaStreamSynchronize(c->stream));
    bool overflow = false;
    int mx = 0;
    for (int p = 0; p < P; ++p) {
        n[p] = (int32_t)c->h_counts[p];
        if (n[p] > cap) overflow = true;
        mx = std::max(mx, std::min(std::min(n[p], cap), g.kp_cap));
    }
    const size_t C = (size_t)g.kp_cap;
    if (mx > 0) {
        if (l_kps) FE_CUDA(c, cudaMemcpy2DAsync(l_kps, sizeof(fe_kpoint) * (size_t)cap, b.lm_lkp, sizeof(fe_kpoint) * C, sizeof(fe_kpoint) * (size_t)mx, P, cudaMemcpyDeviceToHost, c->stream));
        if (r_kps) FE_CUDA(c, cudaMemcpy2DAsync(r_kps, sizeof(fe_kpoint) * (size_t)cap, b.lm_rkp, sizeof(fe_kpoint) * C, sizeof(fe_kpoint) * (size_t)mx, P, cudaMemcpyDeviceToHost, c->stream));
        const size_t row = dim > 0 ? sizeof(float) * dim : binary_bytes(rows);     // descriptor bytes per landmark on the host
        const size_t dev_row = dim > 0 ? row : 32;                                 // and on the device (the float rows are packed)
        const uint8_t *ld = dim > 0 ? reinterpret_cast<const uint8_t *>(b.lm_lfdesc) : b.lm_ldesc;
        const uint8_t *rd = dim > 0 ? reinterpret_cast<const uint8_t *>(b.lm_rfdesc) : b.lm_rdesc;
        for (int s = 0; s < 2; ++s) {
            uint8_t *dst = static_cast<uint8_t *>(s ? r_desc : l_desc);
            const uint8_t *src = s ? rd : ld;
            if (!dst) continue;
            if (row == dev_row) FE_CUDA(c, cudaMemcpy2DAsync(dst, row * cap, src, row * C, row * mx, P, cudaMemcpyDeviceToHost, c->stream));
            else        // BRIEF-16: the leading 16 bytes of every 32-byte device row, pair by pair
                for (int p = 0; p < P; ++p)
                    if (std::min(n[p], mx) > 0)
                        FE_CUDA(c, cudaMemcpy2DAsync(dst + p * row * cap, row, src + p * dev_row * C, dev_row, row, std::min(n[p], mx),
                                                     cudaMemcpyDeviceToHost, c->stream));
        }
        if (matches) FE_CUDA(c, cudaMemcpy2DAsync(matches, sizeof(fe_match) * (size_t)cap, b.lm_match, sizeof(fe_match) * C, sizeof(fe_match) * (size_t)mx, P, cudaMemcpyDeviceToHost, c->stream));
    }
    if ((r = sync_and_resolve(c)) != FE_OK) return r;
    if (overflow) return fail(c, FE_ERR_CAPACITY, "fe_batch_landmarks: more landmarks than capacity");
    return FE_OK;
}

int32_t fe_set_brief_pattern(fe_ctx *c, int32_t bytes, const int8_t *tests, int32_t use_orientation) {
    if (!c || !tests || (bytes != 16 && bytes != 32 && bytes != 64)) return fail(c, FE_ERR_BAD_ARG, "fe_set_brief_pattern: bytes must be 16, 32 or 64");
    for (int i = 0; i < bytes * 8 * 4; ++i)
        if (tests[i] < -24 || tests[i] > 24) return fail(c, FE_ERR_BAD_ARG, "fe_set_brief_pattern: test offsets must lie in [-24, 24] (PATCH_SIZE 48)");
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    const int slot = bytes == 16 ? 0 : bytes == 32 ? 1 : 2;
    const int r = ensure(c, GRP_BRIEF_TAB);
    if (r != FE_OK) return r;
    FE_CUDA(c, cudaMemcpyAsync(c->b.brief_tab + (size_t)slot * 512 * 4, tests, (size_t)bytes * 8 * 4, cudaMemcpyHostToDevice, c->stream));
    FE_CUDA(c, cudaStreamSynchronize(c->stream));
    c->brief_bytes[slot] = bytes;
    c->brief_orient[slot] = use_orientation ? 1 : 0;
    return FE_OK;
}

// cv::FREAK::buildPattern (opencv_contrib xfeatures2d/src/freak.cpp): the table in double, stored as float
int32_t fe_set_freak(fe_ctx *c, int32_t orientation_normalized, int32_t scale_normalized, float pattern_scale, int32_t n_octaves,
                     const int32_t *selected) {
    if (!c) return FE_ERR_BAD_ARG;
    if (!selected)
        return fail(c, FE_ERR_UNSUPPORTED, "fe_set_freak: pass the 512 selected pairs (OpenCV's default FREAK_DEF_PAIRS table is not shipped with this library)");
    if (!(pattern_scale > 0.f) || n_octaves < 1 || n_octaves > 16) return fail(c, FE_ERR_BAD_ARG, "fe_set_freak: pattern_scale > 0, 1 <= n_octaves <= 16");
    constexpr int NS = 64, NO = 256, NP = 43, NPAIRS = 512, NOP = 45;
    for (int i = 0; i < NPAIRS; ++i)
        if (selected[i] < 0 || selected[i] >= NP * (NP - 1) / 2) return fail(c, FE_ERR_BAD_ARG, "fe_set_freak: selected pair index outside [0, 903)");
    const double kPi = 3.1415926535897932384626433832795;
    const int n[8] = {6, 6, 6, 6, 6, 6, 6, 1};
    const double bigR = 2.0 / 3.0, smallR = 2.0 / 24.0, unitSpace = (bigR - smallR) / 21.0;
    const double radius[8] = {bigR, bigR - 6 * unitSpace, bigR - 11 * unitSpace, bigR - 15 * unitSpace, bigR - 18 * unitSpace,
                              bigR - 20 * unitSpace, smallR, 0.0};
    const double sigma[8] = {radius[0] / 2.0, radius[1] / 2.0, radius[2] / 2.0, radius[3] / 2.0, radius[4] / 2.0, radius[5] / 2.0,
                             radius[6] / 2.0, radius[6] / 2.0};
    const double scale_step = std::pow(2.0, (double)n_octaves / NS);
    std::vector<float> tab((size_t)NS * NO * NP * 3);
    for (int s = 0; s < NS; ++s) {
        c->freak_sizes[s] = 0;
        const double sf = std::pow(scale_step, (double)s);
        for (int o = 0; o < NO; ++o) {
            const double theta = double(o) * 2 * kPi / double(NO);
            int p = 0;
            for (int i = 0; i < 8; ++i)
                for (int k = 0; k < n[i]; ++k, ++p) {
                    const double beta = kPi / n[i] * (i % 2);
                    const double alpha = double(k) * 2 * kPi / double(n[i]) + beta + theta;
                    float *e = &tab[(((size_t)s * NO + o) * NP + p) * 3];
                    e[0] = static_cast<float>(radius[i] * std::cos(alpha) * sf * pattern_scale);
                    e[1] = static_cast<float>(radius[i] * std::sin(alpha) * sf * pattern_scale);
                    e[2] = static_cast<float>(sigma[i] * sf * pattern_scale);
                }
        }
        for (int i = 0; i < 8; ++i) {
            const int size_max = static_cast<int>(std::ceil((radius[i] + sigma[i]) * sf * pattern_scale)) + 1;
            if (c->freak_sizes[s] < size_max) c->freak_sizes[s] = size_max;
        }
    }
    // 45 orientation pairs: nine per outer ring (rings 0-3), the three diameters of rings 4-6; integer weights
    int4 op[NOP];
    {
        static const int ring9[9][2] = {{0, 3}, {1, 4}, {2, 5}, {0, 2}, {1, 3}, {2, 4}, {3, 5}, {4, 0}, {5, 1}};
        int m = 0;
        for (int b = 0; b < 24; b += 6)
            for (auto &q : ring9) op[m++] = make_int4(b + q[0], b + q[1], 0, 0);
        for (int b = 24; b < 42; b += 6)
            for (int q = 0; q < 3; ++q) op[m++] = make_int4(b + q, b + q + 3, 0, 0);
        for (m = 0; m < NOP; ++m) {
            const float dx = tab[op[m].x * 3] - tab[op[m].y * 3], dy = tab[op[m].x * 3 + 1] - tab[op[m].y * 3 + 1];
            const float norm_sq = dx * dx + dy * dy;
            op[m].z = int((dx / norm_sq) * 4096.0 + 0.5);
            op[m].w = int((dy / norm_sq) * 4096.0 + 0.5);
        }
    }
    // description pairs = allPairs[selected[k]], allPairs in the order i = 1 .. 42, j = 0 .. i - 1
    uchar2 dp[NPAIRS];
    for (int k = 0; k < NPAIRS; ++k) {
        int i = 1;
        while (i * (i + 1) / 2 <= selected[k]) ++i;
        dp[k] = make_uchar2((unsigned char)i, (unsigned char)(selected[k] - i * (i - 1) / 2));
    }
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    const int r = ensure(c, GRP_FREAK);
    if (r != FE_OK) return r;
    FE_CUDA(c, cudaMemcpyAsync(c->b.freak_tab, tab.data(), tab.size() * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    FE_CUDA(c, cudaMemcpyAsync(c->b.freak_opairs, op, sizeof(op), cudaMemcpyHostToDevice, c->stream));
    FE_CUDA(c, cudaMemcpyAsync(c->b.freak_dpairs, dp, sizeof(dp), cudaMemcpyHostToDevice, c->stream));
    FE_CUDA(c, cudaStreamSynchronize(c->stream));
    c->freak_orient = orientation_normalized ? 1 : 0;
    c->freak_scale_norm = scale_normalized ? 1 : 0;
    c->freak_octaves = n_octaves;
    return FE_OK;
}

int32_t fe_set_chunk_pairs(fe_ctx *c, int32_t pairs) {
    if (!c || pairs < 0) return FE_ERR_BAD_ARG;
    c->chunk_pairs = pairs;
    return FE_OK;
}

int32_t fe_set_batch_descriptor(fe_ctx *c, int32_t desc_kind) {
    if (!c) return FE_ERR_BAD_ARG;
    if (c->hessian)
        return fail(c, FE_ERR_UNSUPPORTED, "fe_set_batch_descriptor: the Fast-Hessian batch describes with SURF (fe_set_batch_detector(ctx, NULL) first)");
    if (desc_kind == FE_DESC_BRIEF64 || desc_kind == FE_DESC_FREAK)
        return fail(c, FE_ERR_UNSUPPORTED, "fe_set_batch_descriptor: the batch matches rows of at most 256 bits (BRIEF-64 / FREAK rows are 512)");
    if (desc_kind == FE_DESC_BRIEF16 || desc_kind == FE_DESC_BRIEF32) {
        if (!c->brief_bytes[brief_slot(desc_kind)])
            return fail(c, FE_ERR_UNSUPPORTED, "fe_set_batch_descriptor: no BRIEF test table of this width (fe_set_brief_pattern)");
    } else if (desc_kind != FE_DESC_ORB256 && desc_dim(desc_kind) == 0) return fail(c, FE_ERR_BAD_ARG, "unknown descriptor kind");
    if (desc_dim(desc_kind) > 0 && detected_surf_win(c) > SURF_DIRECT_MAX_WIN)
        return fail(c, FE_ERR_UNSUPPORTED, "SURF keypoint size not supported");
    c->batch_desc = desc_kind;
    return FE_OK;
}

int32_t fe_set_batch_detector(fe_ctx *c, const fe_surf_params *surf) {
    if (!c) return FE_ERR_BAD_ARG;
    if (!surf) {      // back to FAST / ORB: fe_config, the fe_set_orb_* settings and the batch descriptor were never changed
        c->hessian = false;
        return FE_OK;
    }
    const int nOct = surf->n_octaves > 0 ? surf->n_octaves : 4, nLay = surf->n_octave_layers > 0 ? surf->n_octave_layers : 2;
    if (nOct > 8 || nLay > 8) return fail(c, FE_ERR_BAD_ARG, "fe_set_batch_detector: at most 8 octaves / 8 layers");
    int smem_max = 0;
    FE_CUDA(c, cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, c->cfg.device));
    if (surf_raster_smem(c->cfg.max_keypoints, c->cfg.max_height) > (size_t)smem_max - 1024)
        return fail(c, FE_ERR_UNSUPPORTED, "fe_set_batch_detector: max_keypoints and max_height exceed the raster selection's shared memory");
    c->surf = *surf;
    c->hessian = true;
    return FE_OK;
}

int32_t fe_batch_run(fe_ctx *c, const fe_match_cfg *cfg_a, const fe_match_cfg *cfg_b, int32_t sync) {
    if (!c || c->g.n_images < 2) return fail(c, FE_ERR_BAD_ARG, "fe_batch_run: nothing uploaded");
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    apply_pending_detection(c);
    int r = prepare_batch(c, cfg_a, cfg_b);
    if (r == FE_OK) r = run_batch_on(c, c->g, c->b, c->stream, true, c->g.n_images / 2, cfg_a, cfg_b);
    if (r != FE_OK || !sync) return r;
    if ((r = sync_and_resolve(c)) != FE_OK || !c->hessian) return r;
    // FAST keeps at most kp_cap keypoints, the Fast-Hessian detector may find more maxima than that
    const int NI = c->g.n_images;
    FE_CUDA(c, cudaMemcpyAsync(c->h_counts, c->b.n_kp, sizeof(uint32_t) * NI, cudaMemcpyDeviceToHost, c->stream));
    FE_CUDA(c, cudaStreamSynchronize(c->stream));
    for (int i = 0; i < NI; ++i)
        if ((int)c->h_counts[i] > c->g.kp_cap) return fail(c, FE_ERR_CAPACITY, "fe_batch_run: more Fast-Hessian maxima than fe_config.max_keypoints");
    return FE_OK;
}

int32_t fe_batch_download(fe_ctx *c, int32_t kp_cap, fe_kpoint *kps, uint8_t *desc, int32_t *n_kps,
                          fe_match *ma, int32_t *n_a, fe_match *mb, int32_t *n_b) {
    if (!c || c->g.n_images < 2 || kp_cap < 1) return fail(c, FE_ERR_BAD_ARG, "fe_batch_download: bad argument");
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    const int NP = c->g.n_images / 2;
    bool overflow = false;
    StageTimer t(c, ST_D2H);
    int r = copy_counts(c, 0, NP, c->stream);
    if (r != FE_OK) return r;
    FE_CUDA(c, cudaStreamSynchronize(c->stream));
    if ((r = download_pairs(c, 0, NP, c->stream, {kp_cap, kps, desc, n_kps, ma, n_a, mb, n_b}, overflow)) != FE_OK) return r;
    t.done(0);
    if ((r = sync_and_resolve(c)) != FE_OK) return r;
    if (overflow) return fail(c, FE_ERR_CAPACITY, "fe_batch_download: keypoint capacity exceeded (counts report the required size)");
    return FE_OK;
}

// Pairs per chunk of the overlapped pipeline.  Large enough that one chunk's matcher grid
// (21 CTAs x pairs) still fills the 148 SMs when two chunks are in flight on the two compute lanes.
static int chunk_pairs_init() {
    const char *e = getenv("FE_CHUNK_PAIRS");      // tuning knob; default from measurements on B200
    const int v = e ? atoi(e) : 0;
    return v > 0 ? v : 48;      // gpurun_out/sweep_e2e.log: 48 pairs x 3 host workers = 14.2k pairs/s end to end
}
static const int kChunkPairs = chunk_pairs_init();

static int chunk_pairs_of(const fe_ctx *c) { return c->chunk_pairs > 0 ? c->chunk_pairs : kChunkPairs; }

static int pipeline_chunked(fe_ctx *c, int32_t n_pairs, const uint8_t *left, const uint8_t *right, int32_t w, int32_t h,
                            const fe_match_cfg *cfg_a, const fe_match_cfg *cfg_b, const HostBatch &out) {
    int r = set_geom(c, w, h, 2 * n_pairs);
    if (r != FE_OK) return r;
    apply_pending_detection(c);
    // the chunk views below copy the buffer pointers: everything the batch body reads must exist now
    if ((r = prepare_batch(c, cfg_a, cfg_b)) != FE_OK) return r;
    const Geom &g = c->g;
    const int kChunk = chunk_pairs_of(c);
    const int n_chunks = div_up(n_pairs, kChunk);
    if (!c->s_in) {
        FE_CUDA(c, cudaStreamCreateWithFlags(&c->s_in, cudaStreamNonBlocking));
        FE_CUDA(c, cudaStreamCreateWithFlags(&c->s_out, cudaStreamNonBlocking));
        FE_CUDA(c, cudaStreamCreateWithFlags(&c->s_cmp[0], cudaStreamNonBlocking));
        FE_CUDA(c, cudaStreamCreateWithFlags(&c->s_cmp[1], cudaStreamNonBlocking));
        FE_CUDA(c, cudaEventCreateWithFlags(&c->ev_sync, cudaEventDisableTiming));
    }
    while ((int)c->ev_in.size() < n_chunks) {
        cudaEvent_t a, b;
        FE_CUDA(c, cudaEventCreateWithFlags(&a, cudaEventDisableTiming));
        FE_CUDA(c, cudaEventCreateWithFlags(&b, cudaEventDisableTiming));
        c->ev_in.push_back(a);
        c->ev_done.push_back(b);
    }
    // order the auxiliary streams after whatever is still running on the ctx stream (the zero-fills of prepare_batch included)
    FE_CUDA(c, cudaEventRecord(c->ev_sync, c->stream));
    for (cudaStream_t st : {c->s_in, c->s_out, c->s_cmp[0], c->s_cmp[1]}) FE_CUDA(c, cudaStreamWaitEvent(st, c->ev_sync, 0));

    for (int k = 0; k < n_chunks; ++k) {
        const int p0 = k * kChunk, np = std::min(kChunk, n_pairs - p0);
        // H2D of this chunk's images: left -> even slots, right -> odd slots
        for (int e = 0; e < 2; ++e) {
            const uint8_t *srcp = (e ? right : left) + (size_t)p0 * w * h;
            uint8_t *dstp = c->b.img + (size_t)(2 * p0 + e) * g.img_stride;
            if (g.pitch == w)
                FE_CUDA(c, cudaMemcpy2DAsync(dstp, 2 * g.img_stride, srcp, g.img_stride, g.img_stride, np,
                                             cudaMemcpyHostToDevice, c->s_in));
            else
                for (int i = 0; i < np; ++i)
                    FE_CUDA(c, cudaMemcpy2DAsync(dstp + (size_t)2 * i * g.img_stride, g.pitch, srcp + (size_t)i * w * h, w, w, h,
                                                 cudaMemcpyHostToDevice, c->s_in));
        }
        c->h2d_bytes += (int64_t)2 * np * w * h;
        FE_CUDA(c, cudaEventRecord(c->ev_in[k], c->s_in));
        cudaStream_t cs = c->s_cmp[k & 1];
        FE_CUDA(c, cudaStreamWaitEvent(cs, c->ev_in[k], 0));
        Geom gk = g;
        gk.n_images = 2 * np;
        if ((r = run_batch_on(c, gk, view_of(c->b, g, 2 * p0), cs, false, np, cfg_a, cfg_b)) != FE_OK) return r;
        // counts ride on the compute lane so that the host can size this chunk's downloads
        if ((r = copy_counts(c, p0, np, cs)) != FE_OK) return r;
        FE_CUDA(c, cudaEventRecord(c->ev_done[k], cs));
    }
    bool overflow = false;
    for (int k = 0; k < n_chunks; ++k) {
        const int p0 = k * kChunk, np = std::min(kChunk, n_pairs - p0);
        FE_CUDA(c, cudaEventSynchronize(c->ev_done[k]));
        FE_CUDA(c, cudaStreamWaitEvent(c->s_out, c->ev_done[k], 0));
        if ((r = download_pairs(c, p0, np, c->s_out, out, overflow)) != FE_OK) return r;
    }
    FE_CUDA(c, cudaStreamSynchronize(c->s_out));
    FE_CUDA(c, cudaStreamSynchronize(c->s_in));
    if (take_tc_error(c)) return fail(c, FE_ERR_CUDA, "l2 verification: tcgen05 completion barrier timed out");
    if (overflow) return fail(c, FE_ERR_CAPACITY, "fe_pipeline_batch: keypoint capacity exceeded (counts report the required size)");
    return FE_OK;
}

int32_t fe_pipeline_batch(fe_ctx *c, int32_t n_pairs, const uint8_t *left, const uint8_t *right, int32_t w, int32_t h,
                          const fe_match_cfg *cfg_a, const fe_match_cfg *cfg_b, int32_t kp_cap, fe_kpoint *kps,
                          uint8_t *desc, int32_t *n_kps, fe_match *ma, int32_t *n_a, fe_match *mb, int32_t *n_b) {
    // (the pyramid runs on the whole resident batch; the Fast-Hessian scale space is one per ctx, which two compute lanes
    // would overwrite; every descriptor of the FAST / ORB batch -- ORB-256, BRIEF-16 / 32, SURF -- runs per chunk)
    if (c && left && right && n_pairs >= 2 * chunk_pairs_of(c) && kp_cap >= 1 && c->nlevels == 1 && !c->hessian) {
        // overlapped path: H2D of chunk k+1, kernels of chunk k and D2H of chunk k-1 run concurrently
        FE_CUDA(c, cudaSetDevice(c->cfg.device));
        return pipeline_chunked(c, n_pairs, left, right, w, h, cfg_a, cfg_b, {kp_cap, kps, desc, n_kps, ma, n_a, mb, n_b});
    }
    int r = fe_batch_upload(c, n_pairs, left, right, w, h);
    if (r != FE_OK) return r;
    if ((r = fe_batch_run(c, cfg_a, cfg_b, 0)) != FE_OK) return r;
    return fe_batch_download(c, kp_cap, kps, desc, n_kps, ma, n_a, mb, n_b);
}

int32_t fe_stereo_features(fe_ctx *c, const uint8_t *left, const uint8_t *right, int32_t w, int32_t h, int32_t stride,
                           int32_t desc_kind, fe_kpoint *lk, void *ld, int32_t *nl, fe_kpoint *rk, void *rd, int32_t *nr,
                           int32_t cap, double *proc_seconds) {
    if (!c || !left || !right || !lk || !ld || !nl || !rk || !rd || !nr || cap < 1 || stride < w)
        return fail(c, FE_ERR_BAD_ARG, "fe_stereo_features: bad argument");
    const int dim = desc_dim(desc_kind), bw = brief_width(desc_kind);
    if (desc_kind != FE_DESC_ORB256 && dim == 0 && bw == 0) return fail(c, FE_ERR_UNSUPPORTED, "fe_stereo_features: unknown descriptor kind");
    if (bw > 0 && !c->brief_bytes[brief_slot(desc_kind)])
        return fail(c, FE_ERR_UNSUPPORTED, "fe_stereo_features: no BRIEF test table for this width (fe_set_brief_pattern)");
    FE_CUDA(c, cudaSetDevice(c->cfg.device));
    int r = set_geom(c, w, h, 2);
    if (r != FE_OK) return r;
    const bool upright = c->cfg.surf_upright != 0;
    if (dim > 0) {
        if (detected_surf_win(c) > SURF_DIRECT_MAX_WIN)
            return fail(c, FE_ERR_UNSUPPORTED, "fe_stereo_features: SURF keypoint size not supported");
        if ((r = ensure(c, GRP_FLOAT | (upright ? 0u : GRP_INTEGRAL))) != FE_OK) return r;
    }
    // BRIEF rows: BRIEF-16 / 32 in the 32-byte desc rows, BRIEF-64 in the 64-byte brief_desc rows
    const int brow = bw == 64 ? 64 : 32;
    if (bw > 0 && (r = ensure(c, (bw == 64 ? GRP_BRIEF : 0u) | (c->nlevels > 1 ? GRP_INTEGRAL : 0u))) != FE_OK) return r;
    const bool was = c->profiling;
    c->profiling = true;     // the service reports per-stage ProcTime (bin/feature_node:27-34,72-75)
    { StageTimer t(c, ST_H2D);
      if ((r = upload_images(c, left, 1, stride, 0, 1)) != FE_OK) return r;
      if ((r = upload_images(c, right, 1, stride, 1, 1)) != FE_OK) return r;
      t.done(0); }
    if ((r = run_detect(c, dim == 0 && bw == 0)) != FE_OK) { c->profiling = was; return r; }
    if (dim > 0) {
        StageTimer t(c, ST_SURF);
        t.done(launch_surf(c->g, c->b, c->b.n_kp, dim == 128, upright, detected_surf_win(c), c->stream));
    }
    if (bw > 0 && (r = run_brief_on(c, c->g, c->b, c->stream, true, desc_kind, c->nlevels == 1, bw == 64 ? c->b.brief_desc : c->b.desc,
                                    brow)) != FE_OK) { c->profiling = was; return r; }
    FE_CUDA(c, cudaMemcpyAsync(c->h_counts, c->b.n_kp, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    FE_CUDA(c, cudaStreamSynchronize(c->stream));
    const size_t C = c->g.kp_cap;
    int found[2] = {(int)c->h_counts[0], (int)c->h_counts[1]};
    int kept[2] = {0, 0};
    fe_kpoint *ok[2] = {lk, rk};
    void *od[2] = {ld, rd};
    bool overflow = false;
    for (int e = 0; e < 2; ++e) {
        const int m = std::min(std::min(found[e], cap), (int)C);
        overflow |= found[e] > cap || found[e] > (int)C;
        kept[e] = m;
        if (m > 0) {
            FE_CUDA(c, cudaMemcpyAsync(ok[e], c->b.kp + e * C, sizeof(fe_kpoint) * m, cudaMemcpyDeviceToHost, c->stream));
            if (bw > 0)
                FE_CUDA(c, cudaMemcpy2DAsync(od[e], (size_t)bw, (bw == 64 ? c->b.brief_desc : c->b.desc) + e * C * brow, (size_t)brow,
                                             (size_t)bw, m, cudaMemcpyDeviceToHost, c->stream));
            else if (dim == 0)
                FE_CUDA(c, cudaMemcpyAsync(od[e], c->b.desc + e * C * 32, (size_t)32 * m, cudaMemcpyDeviceToHost, c->stream));
            else
                FE_CUDA(c, cudaMemcpy2DAsync(od[e], sizeof(float) * dim, c->b.fdesc + e * C * 128, sizeof(float) * 128,
                                             sizeof(float) * dim, m, cudaMemcpyDeviceToHost, c->stream));
        }
    }
    r = sync_and_resolve(c);
    c->profiling = was;
    if (r != FE_OK) return r;
    if (dim > 0) {
        // keypoints SURF marked for deletion (size = -1) are removed, src/surf.cpp:953-978
        for (int e = 0; e < 2; ++e) {
            float *d = static_cast<float *>(od[e]);
            int m = 0;
            for (int i = 0; i < kept[e]; ++i)
                if (ok[e][i].size > 0) {
                    if (i > m) { ok[e][m] = ok[e][i]; memmove(d + (size_t)m * dim, d + (size_t)i * dim, sizeof(float) * dim); }
                    ++m;
                }
            if (!overflow) found[e] = m;
        }
    }
    *nl = found[0]; *nr = found[1];
    if (proc_seconds) {
        // both eyes run in the same launches; attribute half of each stage to each eye
        const double det = (c->last_stage_ms[ST_FAST] + c->last_stage_ms[ST_SELECT] + c->last_stage_ms[ST_ORIENT]) * 0.5e-3;
        const double des = (c->last_stage_ms[ST_BLUR] + c->last_stage_ms[ST_BRIEF] + c->last_stage_ms[ST_SURF]) * 0.5e-3;
        proc_seconds[0] = det; proc_seconds[1] = des; proc_seconds[2] = det; proc_seconds[3] = des;
    }
    if (overflow) return fail(c, FE_ERR_CAPACITY, "fe_stereo_features: more keypoints than capacity");
    return FE_OK;
}

}  // extern "C"
