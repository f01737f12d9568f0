// Internal declarations shared by the kernels and the C-ABI layer (not installed).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <atomic>
#include <string>

#include "../../include/fe_abi.h"

namespace fe {

constexpr int STRIP_ROWS = 8;          // FAST strip height of the generic kernel: one CTA = full image width x 8 rows
constexpr int WIDE_STRIP_ROWS = 30;    // strip height of the FAST-9_16 rolling-window kernel (fast16_strip_kernel)
constexpr uint32_t KEY_NONE = 0xFFFFFFFFu;

__host__ __device__ inline int round_up(int v, int m) { return (v + m - 1) / m * m; }
__host__ __device__ inline int div_up(int v, int m) { return (v + m - 1) / m; }

// Geometry of one batch launch (all images of a batch share width/height).
struct Geom {
    int w, h, pitch;       // pitch = round_up(w, 16) bytes
    int n_images;
    int n_strips;          // div_up(h, STRIP_ROWS); also the per-image stride of strip_raw / strip_sel
    int slab_cap;          // candidate capacity per 8-row strip (u32 records)
    size_t slab_img;       // slab records per image: room for either strip layout (see strip_view)
    int kp_cap;            // per-image keypoint capacity
    size_t img_stride;     // bytes between consecutive images (pitch * h)
    int rs_h;              // rows of the row tables (Buffers::rowstart): fe_config.max_height, whatever image is resident
};

// Strip geometry of an image of g.w x g.h (pitch set): shared by set_geom and the pyramid levels.
inline void set_strip_geometry(Geom &g, bool nonmax) {
    g.n_strips = div_up(g.h, STRIP_ROWS);
    g.slab_cap = nonmax ? g.pitch * STRIP_ROWS / 4 : g.pitch * STRIP_ROWS;
    const size_t narrow = (size_t)g.n_strips * (size_t)g.slab_cap;
    const size_t wide = (size_t)div_up(g.h, WIDE_STRIP_ROWS) * (size_t)(g.pitch * WIDE_STRIP_ROWS / 4);
    g.slab_img = narrow > wide ? narrow : wide;
}

struct DetectParams {
    int threshold;         // FAST t
    int ps;                // 16 / 12 / 8
    int nonmax;
    int n_features;        // < 0: keep all
    int edge;              // border filter
    int patch_size;        // ORB patchSize: intensity-centroid disc diameter and rBRIEF pattern
    int wta_k;             // ORB WTA_K
    const int *thr_img = nullptr;   // device, optional: per-image FAST thresholds (grid cells: live_stereo.cpp:293,306)
};

// cv::ORB's steering of a keypoint (orb.cpp): angle = kpt.angle * (float)(CV_PI/180.f), then (float)cos / (float)sin of it
// in double.  Returns (cos, sin).
__device__ __forceinline__ float2 steer(float angle_deg) {
    const float th = __fmul_rn(angle_deg, (float)(3.14159265358979323846 / 180.0));
    return make_float2((float)cos((double)th), (float)sin((double)th));
}

// cv::fastAtan2 (degrees).  Host+device so the exact polynomial can be unit-tested on the CPU.
__host__ __device__ inline float fast_atan2_deg(float y, float x) {
    const float scale = (float)(180.0 / 3.14159265358979323846);
    const float p1 = 0.9997878412794807f * scale, p3 = -0.3258083974640975f * scale,
                p5 = 0.1555786518463281f * scale, p7 = -0.04432655554792128f * scale;
    const float eps = 2.2204460492503131e-16f;
    const float ax = fabsf(x), ay = fabsf(y);
    float a, c, c2;
#ifdef __CUDA_ARCH__
    if (ax >= ay) c = __fdiv_rn(ay, __fadd_rn(ax, eps));
    else c = __fdiv_rn(ax, __fadd_rn(ay, eps));
    c2 = __fmul_rn(c, c);
    a = __fadd_rn(__fmul_rn(p7, c2), p5);
    a = __fadd_rn(__fmul_rn(a, c2), p3);
    a = __fadd_rn(__fmul_rn(a, c2), p1);
    a = __fmul_rn(a, c);
    if (!(ax >= ay)) a = __fsub_rn(90.f, a);
    if (x < 0) a = __fsub_rn(180.f, a);
    if (y < 0) a = __fsub_rn(360.f, a);
#else
    if (ax >= ay) c = ay / (ax + eps);
    else c = ax / (ay + eps);
    c2 = c * c;
    a = p7 * c2; a = a + p5;
    a = a * c2;  a = a + p3;
    a = a * c2;  a = a + p1;
    a = a * c;
    if (!(ax >= ay)) a = 90.f - a;
    if (x < 0) a = 180.f - a;
    if (y < 0) a = 360.f - a;
#endif
    return a;
}

// Exclusive prefix sum of v over a 1024-thread block; total = the block's sum.  s_warp: 33 words of shared memory.
__device__ __forceinline__ uint32_t block_excl_scan_1024(uint32_t v, uint32_t *s_warp, uint32_t &total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t n = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += n;
    }
    if (lane == 31) s_warp[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        uint32_t w = s_warp[lane], wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t n = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += n;
        }
        s_warp[lane] = wi - w;            // exclusive warp bases
        if (lane == 31) s_warp[32] = wi;  // grand total
    }
    __syncthreads();
    const uint32_t r = s_warp[wid] + incl - v;
    total = s_warp[32];
    __syncthreads();
    return r;
}

// ---- keypoints of an image tile (raster-ordered lists: kp_key = y << 16 | x ascending) --------------------------------
// The per-tile kernels (orb_describe_tile_kernel, brief_tile_kernel) find the keypoints of their rows by binary search and
// keep those of their columns by ballot compaction.

// first index in [0, n) whose key is >= target (n if none): 32-way search, one key per lane per round
__device__ __forceinline__ int warp_lower_bound(const uint32_t *__restrict__ keys, int n, uint32_t target, int lane) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int step = (hi - lo + 31) >> 5, i = lo + lane * step;
        const uint32_t m = __ballot_sync(0xffffffffu, i >= hi || keys[i] >= target);
        const int f = m ? __ffs(m) - 1 : 32;          // keys[lo + (f - 1) step] < target <= keys[lo + f step]
        if (f == 0) break;
        hi = min(lo + f * step, hi);
        lo += (f - 1) * step + 1;
    }
    return lo;
}

// Appends the indices and keys of the entries [base, min(base + CHUNK, hi)) whose x lies in [x0, x0 + cols) to s_idx / s_key
// at *s_cnt, in any order (every result of the caller goes to its keypoint's own index).  All THREADS threads call it.
template <int THREADS, int CHUNK>
__device__ __forceinline__ void tile_collect(const uint32_t *keys, int base, int hi, int x0, int cols, uint32_t *s_idx,
                                             uint32_t *s_key, int *s_cnt, int lane) {
#pragma unroll
    for (int q = 0; q < CHUNK / THREADS; ++q) {
        const int i = base + q * THREADS + (int)threadIdx.x;
        uint32_t key = 0;
        bool in = false;
        if (i < hi) {
            key = keys[i];
            in = (int)(key & 0xFFFF) >= x0 && (int)(key & 0xFFFF) < x0 + cols;
        }
        const uint32_t m = __ballot_sync(0xffffffffu, in);
        int pos = 0;
        if (lane == 0 && m) pos = atomicAdd(s_cnt, __popc(m));
        pos = __shfl_sync(0xffffffffu, pos, 0) + __popc(m & ((1u << lane) - 1u));
        if (in) { s_idx[pos] = (uint32_t)i; s_key[pos] = key; }
    }
}

// Warp-cooperative exact FP32 squared L2 distance between a query held in registers (lane l owns dims
// [D/32 * l, D/32 * (l + 1))) and a descriptor row in global memory: coalesced row load, per-lane FMA chain,
// xor-butterfly sum -- a fixed, deterministic summation order; every lane returns the same value.
template <int D>
struct WarpRow {
    float q[D / 32];
    __device__ __forceinline__ void load(const float *row, int lane) {
        if (D == 128) { const float4 v = __ldg(reinterpret_cast<const float4 *>(row) + lane); q[0] = v.x; q[1] = v.y; q[D == 128 ? 2 : 0] = v.z; q[D == 128 ? 3 : 1] = v.w; }
        else { const float2 v = __ldg(reinterpret_cast<const float2 *>(row) + lane); q[0] = v.x; q[1] = v.y; }
    }
    __device__ __forceinline__ float dist2(const float *row, int lane) const {
        float t[D / 32];
        if (D == 128) { const float4 v = __ldg(reinterpret_cast<const float4 *>(row) + lane); t[0] = v.x; t[1] = v.y; t[D == 128 ? 2 : 0] = v.z; t[D == 128 ? 3 : 1] = v.w; }
        else { const float2 v = __ldg(reinterpret_cast<const float2 *>(row) + lane); t[0] = v.x; t[1] = v.y; }
        float acc = 0.f;
#pragma unroll
        for (int i = 0; i < D / 32; ++i) { const float df = __fsub_rn(q[i], t[i]); acc = __fmaf_rn(df, df, acc); }
#pragma unroll
        for (int off = 16; off; off >>= 1) acc = __fadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, off));
        return acc;
    }
};

// ---- device buffers (one set per ctx, sized for cfg.max_*) ------------------------------------
// Largest per-image keypoint capacity the multi-index join of the pruned cross-check serves (match.cu: its shared-memory
// hash table holds 2 x cap x 4 B = 128 KB); above it the join's scratch (cx_half, cx_star) is not allocated.
constexpr int MIH_MAX = 16384;
constexpr int HESSIAN_CHUNK_IMAGES = 8;   // images per scale-space pass of the SURF detector (Buffers::hes_det / hes_trace)

// Layout unit of a buffer: one slice per image, one per pair (image 2p = query/left, 2p+1 = train/right), or one per ctx.
enum BufScope { PER_IMAGE, PER_PAIR, PER_CTX };
// Allocation groups: fe_create allocates GRP_CORE, the paths that need another group allocate it on first use, so that a
// ctx never pays for memory its descriptors and matchers do not read.
enum BufGroup : unsigned {
    GRP_CORE = 1u << 0,        // detection, ORB-256 descriptors, Hamming matching
    GRP_FLOAT = 1u << 1,       // float descriptors (SURF) and L2 matching
    GRP_INTEGRAL = 1u << 2,    // integral images (SURF orientation, BRIEF, FREAK)
    GRP_VERIFY = 1u << 3,      // exact tensor-core L2 cross-check (l2verify.cu)
    GRP_CROSS = 1u << 4,       // pruned Hamming cross-check
    GRP_HARRIS = 1u << 5,      // cv::ORB HARRIS_SCORE
    GRP_BRIEF = 1u << 6,       // 64-byte binary rows (BRIEF-16 / 32 / 64, FREAK)
    GRP_BRIEF_TAB = 1u << 7,   // cv::BriefDescriptorExtractor test tables
    GRP_FREAK = 1u << 8,       // cv::FREAK pattern
    GRP_WINDOW = 1u << 9,      // WindowMatcher over a resident sequence (fe_window_batch)
    GRP_WLIVE = 1u << 10,      // its liveGraph variant: right-descriptor cross-check
    GRP_WUPDATE = 1u << 11,    // fe_window_update's current / previous landmark lists
    GRP_SURFDET = 1u << 12,    // Fast-Hessian scale space
    GRP_LANDMARKS = 1u << 13,  // stereoLandmarks packing
    GRP_PYRAMID = 1u << 14,    // multi-level ORB
    GRP_WFLOAT = 1u << 15,     // WindowMatcher over a resident SURF sequence: float landmark rows, 64-bit L2 keys
    GRP_WFLIVE = 1u << 16,     // its liveGraph variant: right float rows and the right side's keys
    GRP_WUFLOAT = 1u << 17,    // fe_window_update's current / previous float rows (SURF-64 / SURF-128)
    GRP_LMFLOAT = 1u << 18,    // stereoLandmarks packing of SURF batches
};

// Every device buffer of a ctx, declared once: X(element type, name, scope, group, elements per unit).  The element count is
// an expression of the Geom `g`: at the capacity geometry (fe_config.max_*) it sizes the allocation, at the resident geometry
// it is the stride by which a view of images [first, ...) offsets the buffer.  Buffers, allocation, views and teardown are
// all generated from this list.
#define FE_BUFFERS(X) \
    X(uint8_t, img, PER_IMAGE, GRP_CORE, g.img_stride)             /* [h][pitch] */ \
    X(uint8_t, blur, PER_IMAGE, GRP_CORE, g.img_stride)            /* same layout */ \
    X(uint8_t, respmap, PER_IMAGE, GRP_CORE, g.img_stride)         /* same layout: NMS-surviving FAST responses (s - t), 0 elsewhere */ \
    X(uint32_t, slab, PER_IMAGE, GRP_CORE, g.slab_img)             /* per strip (StripView) records score<<24 | ylocal<<16 | x */ \
    X(uint32_t, strip_raw, PER_IMAGE, GRP_CORE, g.n_strips)        /* candidates emitted per strip */ \
    X(uint32_t, strip_sel, PER_IMAGE, GRP_CORE, g.n_strips)        /* survivors of the top-N cut per strip */ \
    X(uint32_t, hist, PER_IMAGE, GRP_CORE, 256)                    /* response histogram (inside the border) */ \
    X(uint32_t, n_kp, PER_IMAGE, GRP_CORE, 1)                      /* keypoints found (may exceed kp_cap) */ \
    X(uint32_t, n_override, PER_IMAGE, GRP_CORE, 1)                /* counts for externally supplied kps */ \
    X(int, thr_img, PER_IMAGE, GRP_CORE, 1)                        /* per-image FAST thresholds (grid detector) */ \
    X(int, rowstart, PER_IMAGE, GRP_CORE, g.rs_h + 2)              /* first keypoint whose floor(y) >= row (raster-ordered lists) */ \
    X(int8_t, pattern, PER_CTX, GRP_CORE, 1024)                    /* [512][2] rBRIEF points when patch size != 31 or WTA_K != 2 (else the built-in table) */ \
    X(int, umax, PER_CTX, GRP_CORE, 128)                           /* OpenCV's umax table of the general orientation kernel */ \
    X(uint32_t, kp_key, PER_IMAGE, GRP_CORE, g.kp_cap)             /* (y<<16 | x), ascending = raster order */ \
    X(uint8_t, kp_score, PER_IMAGE, GRP_CORE, g.kp_cap) \
    X(fe_kpoint, kp, PER_IMAGE, GRP_CORE, g.kp_cap)                /* wire layout */ \
    X(float, kx, PER_IMAGE, GRP_CORE, g.kp_cap) \
    X(float, ky, PER_IMAGE, GRP_CORE, g.kp_cap) \
    X(float2, kcs, PER_IMAGE, GRP_CORE, g.kp_cap)                  /* (cos, sin) of the steering angle */ \
    X(uint8_t, desc, PER_IMAGE, GRP_CORE, 32 * g.kp_cap) \
    X(uint32_t, best, PER_PAIR, GRP_CORE, g.kp_cap)                /* matching keys (distance << 16 | index) */ \
    X(uint32_t, second, PER_PAIR, GRP_CORE, g.kp_cap) \
    X(uint32_t, allbest, PER_PAIR, GRP_CORE, g.kp_cap) \
    X(uint32_t, colbest, PER_PAIR, GRP_CORE, g.kp_cap) \
    X(fe_match, match_a, PER_PAIR, GRP_CORE, g.kp_cap) \
    X(fe_match, match_b, PER_PAIR, GRP_CORE, g.kp_cap) \
    X(uint32_t, n_a, PER_PAIR, GRP_CORE, 1) \
    X(uint32_t, n_b, PER_PAIR, GRP_CORE, 1) \
    X(float, fdesc, PER_IMAGE, GRP_FLOAT, 128 * g.kp_cap)          /* rows of 128 floats (SURF-64 uses the first 64) */ \
    X(unsigned long long, best64, PER_PAIR, GRP_FLOAT, g.kp_cap)   /* L2 keys: float bits of d^2 << 32 | index */ \
    X(unsigned long long, second64, PER_PAIR, GRP_FLOAT, g.kp_cap) \
    X(unsigned long long, allbest64, PER_PAIR, GRP_FLOAT, g.kp_cap) \
    X(unsigned long long, colbest64, PER_PAIR, GRP_FLOAT, g.kp_cap) \
    X(uint16_t, bf16desc, PER_IMAGE, GRP_FLOAT, round_up(div_up(g.kp_cap, 128), 2) * 128 * 160)  /* bf16 UMMA operands: [tiles][dim/8 + 4][128][8] */ \
    X(float, fnorm, PER_IMAGE, GRP_FLOAT, round_up(div_up(g.kp_cap, 128), 2) * 128)             /* |x|^2 per row: [tiles * 128] */ \
    X(uint32_t, cand, PER_PAIR, GRP_FLOAT, 8 * g.kp_cap)           /* [2][kp_cap][4] per-row candidates */ \
    X(int, tc_error, PER_CTX, GRP_FLOAT, 1)                        /* tcgen05 completion-barrier timeout flag */ \
    X(int32_t, integral, PER_IMAGE, GRP_INTEGRAL, (size_t)(g.h + 1) * (g.w + 1))   /* CV_32S integral image */ \
    X(unsigned long long, vf_candL, PER_PAIR, GRP_VERIFY, g.kp_cap)   /* band candidates */ \
    X(unsigned long long, vf_candR, PER_PAIR, GRP_VERIFY, g.kp_cap) \
    X(float, vf_limq, PER_PAIR, GRP_VERIFY, round_up(g.kp_cap, 128))  /* thresholds */ \
    X(float, vf_limt, PER_PAIR, GRP_VERIFY, round_up(g.kp_cap, 128)) \
    X(float, vf_limqd, PER_PAIR, GRP_VERIFY, round_up(g.kp_cap, 128)) \
    X(float, vf_limtd, PER_PAIR, GRP_VERIFY, round_up(g.kp_cap, 128)) \
    X(uint32_t, vf_list, PER_PAIR, GRP_VERIFY, l2_verify_list_entries(g.kp_cap))   /* flagged-element lists */ \
    X(uint32_t, vf_npush, PER_PAIR, GRP_VERIFY, 1) \
    X(uint32_t, vf_maxnorm, PER_IMAGE, GRP_VERIFY, 1) \
    X(uint32_t, cx_bestL, PER_PAIR, GRP_CROSS, g.kp_cap)           /* band candidates */ \
    X(uint32_t, cx_bestR, PER_PAIR, GRP_CROSS, g.kp_cap) \
    X(uint32_t, cx_dummy, PER_PAIR, GRP_CROSS, g.kp_cap) \
    X(int, cx_thrq, PER_PAIR, GRP_CROSS, g.kp_cap)                 /* thresholds */ \
    X(int, cx_thrt, PER_PAIR, GRP_CROSS, g.kp_cap) \
    X(uint16_t, cx_qperm, PER_PAIR, GRP_CROSS, g.kp_cap)           /* easy / hard partitions */ \
    X(uint16_t, cx_tperm, PER_PAIR, GRP_CROSS, g.kp_cap) \
    X(uint32_t, cx_n, PER_PAIR, GRP_CROSS, 8)                      /* class sizes A, B, C of the queries, then of the trains */ \
    X(uint16_t, cx_half, PER_PAIR, GRP_CROSS, g.kp_cap <= MIH_MAX ? 32 * g.kp_cap : 0)   /* [2][16][kp_cap] halves in permutation order */ \
    X(uint16_t, cx_star, PER_PAIR, GRP_CROSS, g.kp_cap <= MIH_MAX ? 2 * g.kp_cap : 0)    /* [2][kp_cap] own candidate */ \
    X(float, harris, PER_IMAGE, GRP_HARRIS, g.kp_cap)              /* Harris responses */ \
    X(uint8_t, brief_desc, PER_IMAGE, GRP_BRIEF, 64 * g.kp_cap)    /* rows 64 bytes apart */ \
    X(int8_t, brief_tab, PER_CTX, GRP_BRIEF_TAB, 3 * 512 * 4)      /* [BRIEF-16 / 32 / 64][bytes * 8][4] (y1, x1, y2, x2) tests */ \
    X(float, freak_tab, PER_CTX, GRP_FREAK, 64 * 256 * 43 * 3)     /* [scale][orientation][point] (x, y, sigma) */ \
    X(int4, freak_opairs, PER_CTX, GRP_FREAK, 45)                  /* (i, j, weight_dx, weight_dy) */ \
    X(uchar2, freak_dpairs, PER_CTX, GRP_FREAK, 512)               /* (i, j) */ \
    X(int32_t, freak_scale, PER_IMAGE, GRP_FREAK, g.kp_cap)        /* scale index per keypoint */ \
    /* WindowMatcher sequence: landmark lists as virtual pairs (cur = slot 2v, prev = slot 2v + 1) */ \
    X(uint8_t, wdesc, PER_IMAGE, GRP_WINDOW, 32 * g.kp_cap) \
    X(float, wkx, PER_IMAGE, GRP_WINDOW, g.kp_cap) \
    X(float, wky, PER_IMAGE, GRP_WINDOW, g.kp_cap) \
    X(uint32_t, wcount, PER_IMAGE, GRP_WINDOW, 1) \
    X(uint32_t, wbest, PER_PAIR, GRP_WINDOW, g.kp_cap) \
    X(uint32_t, wsecond, PER_PAIR, GRP_WINDOW, g.kp_cap) \
    X(fe_match, wmatch, PER_PAIR, GRP_WINDOW, g.kp_cap) \
    X(uint32_t, wn, PER_PAIR, GRP_WINDOW, 1) \
    X(double, wq, PER_CTX, GRP_WINDOW, 16) \
    X(double, wxyz, PER_PAIR, GRP_WINDOW, 3 * g.kp_cap) \
    X(uint8_t, wdesc_r, PER_IMAGE, GRP_WLIVE, 32 * g.kp_cap)       /* right descriptors of the landmarks */ \
    X(uint32_t, wbest_r, PER_PAIR, GRP_WLIVE, g.kp_cap)            /* row / column arg-mins of the right-descriptor cross-check */ \
    X(uint32_t, wcol_r, PER_PAIR, GRP_WLIVE, g.kp_cap) \
    /* the same window over a SURF sequence: float rows at fdesc's 128-float stride, L2 keys (float bits of d^2 << 32 | index) */ \
    X(float, wfdesc, PER_IMAGE, GRP_WFLOAT, 128 * g.kp_cap) \
    X(unsigned long long, wbest64, PER_PAIR, GRP_WFLOAT, g.kp_cap)        /* row best (ratio) / row arg-min (cross-check) */ \
    X(unsigned long long, wsecond64, PER_PAIR, GRP_WFLOAT, g.kp_cap)      /* row second (ratio) / column arg-min (cross-check) */ \
    X(float, wfdesc_r, PER_IMAGE, GRP_WFLIVE, 128 * g.kp_cap)            /* right float rows of the landmarks */ \
    X(unsigned long long, wbest64_r, PER_PAIR, GRP_WFLIVE, g.kp_cap)      /* row / column arg-mins of the right-row cross-check */ \
    X(unsigned long long, wcol64_r, PER_PAIR, GRP_WFLIVE, g.kp_cap) \
    /* fe_window_update: the current (slot 0) and previous (slot 1) frame's landmark lists */ \
    X(fe_kpoint, wu_kp, PER_CTX, GRP_WUPDATE, 2 * g.kp_cap) \
    X(uint8_t, wu_desc, PER_CTX, GRP_WUPDATE, 64 * g.kp_cap) \
    X(uint8_t, wu_rdesc, PER_CTX, GRP_WUPDATE, 64 * g.kp_cap) \
    X(float, wu_kx, PER_CTX, GRP_WUPDATE, 2 * g.kp_cap) \
    X(float, wu_ky, PER_CTX, GRP_WUPDATE, 2 * g.kp_cap) \
    X(float2, wu_kcs, PER_CTX, GRP_WUPDATE, 2 * g.kp_cap)          /* scratch of the keypoint unpack */ \
    X(uint32_t, wu_n, PER_CTX, GRP_WUPDATE, 2) \
    X(float, wu_fdesc, PER_CTX, GRP_WUFLOAT, 2 * 128 * g.kp_cap)        /* [2][kp_cap][128] left float rows */ \
    X(float, wu_frdesc, PER_CTX, GRP_WUFLOAT, 2 * 128 * g.kp_cap)       /* [2][kp_cap][128] right float rows */ \
    /* Fast-Hessian scale space: [image of the pass][all layers back to back] */ \
    X(float, hes_det, PER_CTX, GRP_SURFDET, (size_t)std::min(g.n_images, HESSIAN_CHUNK_IMAGES) * g.w * g.h * 20) \
    X(float, hes_trace, PER_CTX, GRP_SURFDET, (size_t)std::min(g.n_images, HESSIAN_CHUNK_IMAGES) * g.w * g.h * 20) \
    X(uint32_t, hes_count, PER_CTX, GRP_SURFDET, 2 * g.n_images)   /* [n_images] accepted maxima, then [n_images] largest size (float bits) */ \
    X(fe_kpoint, hes_kp, PER_IMAGE, GRP_SURFDET, g.kp_cap)         /* unsorted maxima */ \
    X(fe_kpoint, lm_lkp, PER_PAIR, GRP_LANDMARKS, g.kp_cap) \
    X(fe_kpoint, lm_rkp, PER_PAIR, GRP_LANDMARKS, g.kp_cap) \
    X(uint8_t, lm_ldesc, PER_PAIR, GRP_LANDMARKS, 32 * g.kp_cap) \
    X(uint8_t, lm_rdesc, PER_PAIR, GRP_LANDMARKS, 32 * g.kp_cap) \
    X(fe_match, lm_match, PER_PAIR, GRP_LANDMARKS, g.kp_cap) \
    X(float, lm_lfdesc, PER_PAIR, GRP_LMFLOAT, 128 * g.kp_cap)          /* rows of dim floats, packed (the host's layout) */ \
    X(float, lm_rfdesc, PER_PAIR, GRP_LMFLOAT, 128 * g.kp_cap) \
    /* multi-level ORB: two ping-pong level images (level-1 geometry is the largest), coefficient table, accumulated results */ \
    X(uint8_t, pyr_img0, PER_IMAGE, GRP_PYRAMID, g.img_stride) \
    X(uint8_t, pyr_img1, PER_IMAGE, GRP_PYRAMID, g.img_stride) \
    X(int, pyr_tab, PER_CTX, GRP_PYRAMID, 2 * (g.w + g.h)) \
    X(fe_kpoint, pyr_kp, PER_IMAGE, GRP_PYRAMID, g.kp_cap) \
    X(uint8_t, pyr_desc, PER_IMAGE, GRP_PYRAMID, 32 * g.kp_cap) \
    X(uint32_t, pyr_n, PER_IMAGE, GRP_PYRAMID, 1)

struct Buffers {
#define FE_BUFFER_FIELD(T, name, scope, group, n) T *name = nullptr;
    FE_BUFFERS(FE_BUFFER_FIELD)
#undef FE_BUFFER_FIELD
};

// The strip layout the FAST kernel of this (geometry, parameters) writes and the top-N selection reads: strip s of an image
// starts at slab + image * g.slab_img + s * cap and holds its candidates in raster order (ylocal < rows).
struct StripView { int rows, n, cap; };
StripView strip_view(const Geom &g, const DetectParams &p);

// ---- kernel launchers (each returns the number of kernels it launched) -------------------------
int launch_fast(const Geom &g, const DetectParams &p, const Buffers &b, cudaStream_t s);
int launch_select(const Geom &g, const DetectParams &p, const Buffers &b, cudaStream_t s);
// Wire keypoints, kx / ky and the steering of the selected keypoints; with orientation, the intensity-centroid angle of
// p.patch_size (the kernel follows from p.patch_size and p.edge, orb.cu)
int launch_orient(const Geom &g, const DetectParams &p, const Buffers &b, bool orientation, cudaStream_t s);
int launch_blur(const Geom &g, const Buffers &b, cudaStream_t s);
// Whether launch_describe_tile serves the geometry of p (patch size, edgeThreshold, WTA_K).  The caller still requires
// orientation, descriptors and the FAST score.
bool describe_tile_fits(const DetectParams &p);
// orientation + wire keypoints + rBRIEF-256 per image tile, from b.img and b.blur: writes what launch_orient and launch_rbrief
// write
int launch_describe_tile(const Geom &g, const DetectParams &p, const Buffers &b, cudaStream_t s);
// cv::ORB HARRIS_SCORE (harris.cu): score the selected FAST corners, keep the n_features best (ties kept, raster order);
// then, after the keypoints are packed, store the score as their response
int launch_harris_select(const Geom &g, int n_features, const Buffers &b, cudaStream_t s);
int launch_harris_store(const Geom &g, const Buffers &b, cudaStream_t s);

// cv::cornerSubPix (win x win half-size, zeroZone -1) for the keypoints of every image of the batch.
// Sampling image of batch image i: src[i] (w[i] x h[i], row pitch[i]); the point is  (kp + pre) -> refine ->
// (+ post1) + post2  with float adds in that order (src/live_stereo.cpp:321-350, features.py:623-640).
constexpr int SUBPIX_MAX_IMAGES = 16;
struct SubpixParams {
    const uint8_t *src[SUBPIX_MAX_IMAGES];
    int w[SUBPIX_MAX_IMAGES], h[SUBPIX_MAX_IMAGES], pitch[SUBPIX_MAX_IMAGES];
    float pre_x[SUBPIX_MAX_IMAGES], pre_y[SUBPIX_MAX_IMAGES];
    float post1_x[SUBPIX_MAX_IMAGES], post1_y[SUBPIX_MAX_IMAGES], post2_x[SUBPIX_MAX_IMAGES], post2_y[SUBPIX_MAX_IMAGES];
    int refine;              // 0: only apply the offsets
    int max_iters;           // 40
    float epsilon;           // 0.001
};
int launch_subpix(const Geom &g, const Buffers &b, const uint32_t *counts, const SubpixParams &sp, cudaStream_t s);
// ORB descriptors of the keypoints in b.kx / b.ky / b.kcs from b.blur (and b.img outside the image): rBRIEF-256 for WTA_K 2,
// 128 tuples of WTA_K points from b.pattern otherwise (the kernel follows from p.patch_size, p.edge and p.wta_k, orb.cu)
int launch_rbrief(const Geom &g, const DetectParams &p, const Buffers &b, const uint32_t *counts, cudaStream_t s);
int launch_unpack_kps(const Geom &g, const Buffers &b, const uint32_t *counts, cudaStream_t s);
// cv::BriefDescriptorExtractor(bytes) at the keypoints in b.kp with the caller's test table (brief.cu); needs b.integral.
// out rows are row_bytes apart (>= bytes; the rest of a row is zeroed)
int launch_brief_ext(const Geom &g, const Buffers &b, const uint32_t *counts, const int8_t *pattern, int bytes, int use_orientation,
                     uint8_t *out, int row_bytes, cudaStream_t s);
// The same rows from b.img per image tile, for the raster-ordered keypoints of one level (b.kp_key, b.n_kp) that all lie 28 px
// inside the image (launch_brief_border first)
int launch_brief_tile(const Geom &g, const Buffers &b, const int8_t *pattern, int bytes, int use_orientation, uint8_t *out,
                      int row_bytes, cudaStream_t s);
// BriefDescriptorExtractor::compute's runByImageBorder(28) on the detected keypoints: keeps them in order and compacts b.kp,
// b.kp_key, b.kx, b.ky; b.n_kp becomes the kept count
int launch_brief_border(const Geom &g, const Buffers &b, cudaStream_t s);

// cv::FREAK at the keypoints in b.kp (freak.cu); needs b.integral and b.img.  table: [64][256][43] (x, y, sigma); opairs: [45]
// (i, j, weight_dx, weight_dy); dpairs: [512] (i, j); scale_idx: [n_images][kp_cap].  Writes kp.angle and 64-byte rows.
int launch_freak(const Geom &g, const Buffers &b, const uint32_t *counts, const int32_t *scale_idx, const float *table,
                 const int4 *opairs, const uchar2 *dpairs, int orientation_normalized, uint8_t *out, cudaStream_t s);

// SURF / SURF_EXTENDED descriptors at the keypoints in b.kp (x, y, size); writes b.fdesc rows of
// `128` floats (64 used when !extended), kp.angle, and kp.size = -1 for keypoints the reference drops.
// max_win: upper bound of (int)(21 * size * 1.2 / 9) over the batch's keypoints (picks the shared-memory variant).
int launch_surf(const Geom &g, const Buffers &b, const uint32_t *counts, bool extended, bool upright, int max_win,
                cudaStream_t s);
constexpr int SURF_DIRECT_MAX_WIN = 1024;   // windows above SURF_MAX_WIN are produced on the fly (never staged), up to this size
constexpr int SURF_MAX_WIN = 88;   // largest supported (int)(21 * size * 1.2 / 9): keypoint size <= 31.4 (ORB: 31 -> 86)
constexpr int SURF_ORI_RADIUS = 6;  // orientation samples: the (i, j) with i^2 + j^2 <= 36

// Scale of a SURF keypoint (src/surf.cpp:609-611): s = size * 1.2 / 9, the Haar wavelet size and the descriptor window.
struct SurfScale { float s; int grad_wav_size, win_size; };
__device__ __forceinline__ SurfScale surf_scale(float size) {
    SurfScale r;
    r.s = __fdiv_rn(__fmul_rn(size, 1.2f), 9.0f);
    r.grad_wav_size = 2 * __float2int_rn(__fmul_rn(2.f, r.s));
    r.win_size = (int)__fmul_rn(21.f, r.s);
    return r;
}

// Orientation sample (i, j) of a keypoint at (cx, cy): its Haar wavelet's top-left corner (x, y) on the integral image and
// whether the wavelet lies inside the w x h image (src/surf.cpp:630-636).  half = (grad_wav_size - 1) / 2.
__device__ __forceinline__ bool surf_ori_sample(float cx, float cy, const SurfScale &sc, float half, int i, int j, int w, int h,
                                                int &x, int &y) {
    x = __float2int_rn(__fsub_rn(__fadd_rn(cx, __fmul_rn((float)i, sc.s)), half));
    y = __float2int_rn(__fsub_rn(__fadd_rn(cy, __fmul_rn((float)j, sc.s)), half));
    return !(y < 0 || y >= (h + 1) - sc.grad_wav_size || x < 0 || x >= (w + 1) - sc.grad_wav_size);
}

// SURFInvoker's drop rule (src/surf.cpp:953-978): the keypoints whose descriptor the reference does not compute and which it
// removes.  Geometric only: the wavelet larger than the image, a window outside [1, max_win], or -- oriented -- no orientation
// sample inside the image.  The descriptor kernel and the batch's raster selection of Fast-Hessian maxima both decide with it,
// so a batch never holds a keypoint the descriptor pass drops.
__device__ __forceinline__ bool surf_drops(float cx, float cy, float size, int w, int h, bool upright, int max_win) {
    const SurfScale sc = surf_scale(size);
    if (h + 1 < sc.grad_wav_size || w + 1 < sc.grad_wav_size || sc.win_size < 1 || sc.win_size > max_win) return true;
    if (upright) return false;
    const float half = __fdiv_rn((float)(sc.grad_wav_size - 1), 2.f);
    for (int i = -SURF_ORI_RADIUS; i <= SURF_ORI_RADIUS; ++i)
        for (int j = -SURF_ORI_RADIUS; j <= SURF_ORI_RADIUS; ++j) {
            int x, y;
            if (i * i + j * j <= SURF_ORI_RADIUS * SURF_ORI_RADIUS && surf_ori_sample(cx, cy, sc, half, i, j, w, h, x, y)) return false;
        }
    return true;
}

// multi-level ORB (pyramid.cu)
int launch_resize_linear_exact(const uint8_t *src, int sw, int sh, int spitch, size_t sstride, uint8_t *dst, int dw, int dh,
                               int dpitch, size_t dstride, const int *tab, int n_images, cudaStream_t s);
int launch_pyr_append(const Geom &g, int level, float scale, float kp_size, const Buffers &b, fe_kpoint *akp, uint8_t *adesc,
                      uint32_t *n_acc, bool with_desc, cudaStream_t s);
int launch_pyr_coords(const Geom &g, const Buffers &b, cudaStream_t s);

// SURF Fast-Hessian detector (surf_detect.cu)
struct HaarBoxI { int dx1, dy1, dx2, dy2; float w; };
struct HessianLayer {
    int size, step, margin, samples_i, samples_j, valid;
    HaarBoxI box[10];          // 3 Dxx, 3 Dyy, 4 Dxy boxes of the 9 x 9 pattern resized to `size`
};
// all three take a batch of n_images (blockIdx.z / .y): image i reads S + i * s_img_stride, layer arrays det + i * l_img_stride
int launch_hessian_layer(const int32_t *S, size_t s_img_stride, int stride, int R, int C, const HessianLayer &hl, float *det,
                         float *trace, size_t l_img_stride, int n_images, cudaStream_t s);
int launch_hessian_maxima(const float *d0, const float *d1, const float *d2, const float *tr, size_t l_img_stride, int rows,
                          int cols, int margin, int size, int size_prev, int step, int octave, float threshold, fe_kpoint *out,
                          int cap, uint32_t *count, int n_images, cudaStream_t s);
// std::sort(keypoints, KeypointGreater()) on the device; also the largest keypoint size per image (float bits)
int launch_surf_rank_sort(const fe_kpoint *in, fe_kpoint *out, const uint32_t *count, int cap, uint32_t *max_size_bits, int n_images,
                          cudaStream_t s);
int launch_integral(const Geom &g, const Buffers &b, cudaStream_t s);
// Batched pipeline (fe_set_batch_detector): of the count[i] maxima in in + i * kp_cap, those SURFInvoker keeps
// (surf_drops), in raster order (y, x, then KeypointGreater) -> b.kp, b.kx, b.ky; b.n_kp = survivors, or the maxima count when
// it exceeds kp_cap.  One CTA per image of g, surf_raster_smem(kp_cap, h) bytes of dynamic shared memory.
size_t surf_raster_smem(int kp_cap, int h);
int launch_surf_raster(const Geom &g, const fe_kpoint *in, const uint32_t *count, bool upright, const Buffers &b, cudaStream_t s);

// WindowMatcher over a resident sequence (window.cu)
// side 0: left keypoints / descriptors of the landmarks (queryIdx of matches_a); side 1: right descriptors (trainIdx), wkx / wky unused
int launch_gather_landmarks(const Geom &g, int n_frames, const Buffers &b, int side, uint8_t *wdesc, float *wkx, float *wky,
                            uint32_t *wcount, cudaStream_t s);
// SURF batches: the first dim (64 / 128) floats of the b.fdesc rows, to rows of 128 floats in wfdesc
int launch_gather_landmarks(const Geom &g, int n_frames, const Buffers &b, int side, int dim, float *wfdesc, float *wkx,
                            float *wky, uint32_t *wcount, cudaStream_t s);
int launch_triangulate(const Geom &g, int n_frames, const Buffers &b, const double *Q, double *xyz, cudaStream_t s);
int launch_pack_landmarks(const Geom &g, int n_pairs, const Buffers &b, const uint32_t *n_m, const fe_match *matches,
                          fe_kpoint *lkp, fe_kpoint *rkp, uint8_t *ldesc, uint8_t *rdesc, fe_match *out, cudaStream_t s);
// SURF batches: rows of dim floats, packed (dim floats apart)
int launch_pack_landmarks(const Geom &g, int n_pairs, const Buffers &b, const uint32_t *n_m, const fe_match *matches,
                          fe_kpoint *lkp, fe_kpoint *rkp, int dim, float *ldesc, float *rdesc, fe_match *out, cudaStream_t s);

// Row table of raster-ordered keypoint lists (match.cu): rowstart[image][r] = first index whose floor(y), clamped to
// [0, h], is >= r, for r in [0, h + 1] (rowstart[h + 1] = n); h = Geom::rs_h.  The banded matchers read their candidate range from it instead of searching.
int launch_rowstart(const Geom &g, const Buffers &b, const uint32_t *counts, cudaStream_t s);
// Candidate index range [lo, hi) of a query whose allowed trains have raw y within `reach` of c (one row of slack on both
// sides for float rounding; the caller still applies the exact predicate).
__device__ __forceinline__ void band_range(const int *rows, int h, float c, float reach, int &lo, int &hi) {
    const int r0 = (int)floorf(c - reach) - 1, r1 = (int)floorf(c + reach) + 2;
    lo = rows[min(max(r0, 0), h)];          // rows 0 and h also hold the keypoints whose y was clamped into the table
    hi = rows[min(max(r1, 1), h + 1)];
}

// Trim the table's candidate range to the exact allowed run with warp-wide ballots from both ends (keypoint y is
// non-decreasing, so `started(t)` -- t is at or after the first allowed index -- and `past(t)` -- t is beyond the last one --
// are monotone false -> true).  One round per end unless a row holds more than 32 keypoints in the slack.
template <typename PA, typename PB>
__device__ __forceinline__ void band_trim(int &lo, int &hi, int lane, PA started, PB past) {
    while (lo < hi) {
        const int t = lo + lane;
        const uint32_t m = __ballot_sync(0xffffffffu, t < hi ? started(t) : true);
        if (m) { lo = min(lo + __ffs(m) - 1, hi); break; }
        lo += 32;
    }
    while (hi > lo) {
        const int t = hi - 32 + lane;
        const uint32_t m = __ballot_sync(0xffffffffu, t >= lo ? past(t) : false);
        if (m == 0) break;
        hi = hi - 32 + __ffs(m) - 1;                       // first index of this window that is past the run
        if (m != 0xffffffffu) break;                       // (all 32 past: look at the window before it)
    }
}

struct MatchParams {
    int mask;                  // fe_mask_kind for the (best, second) pair
    float epi_threshold, q_off, t_off;
    float half_w, half_h;
    int h2 = 0;                // 1: cv::NORM_HAMMING2 (two-bit symbols, ORB WTA_K 3 / 4)
};
// unmasked row arg-min + column arg-min (cross-check)
// register-only POPC throughput probe; returns the number of POPCs issued
double launch_popc_peak(int sms, int iters, uint32_t *sink, cudaStream_t s);
int launch_hamming_cross(const Geom &g, int n_pairs, bool h2, const Buffers &b, const uint32_t *counts, cudaStream_t s);
// cross-check + |dy| <= max_dy by band candidates + pruned verification (raster-ordered keypoints on both sides);
// writes match_b / n_b itself (no separate finalize).  row_bytes: 32, or 16 for 128-bit rows zero-padded in the 256-bit rows
// (the multi-index join then reads only their 8 data halves)
// fused_ratio >= 0: mode A's Lowe-ratio finalize (b.best / b.second -> match_a / n_a) rides in the same finalize launch
int launch_hamming_cross_pruned(const Geom &g, int n_pairs, float max_dy, bool have_band, bool use_join, int row_bytes, const Buffers &b,
                                const uint32_t *counts, double fused_ratio, cudaStream_t s, cudaStream_t aux = nullptr,
                                cudaEvent_t ev_fork = nullptr, cudaEvent_t ev_join = nullptr);      // aux: side stream for the join
// masked kNN-2; train_sorted = train keypoints are in raster order (enables the banded kernel)
// inner_thr >= 0 (epipolar band path only): additionally produce the cross-check's band candidates b.cx_bestL / b.cx_bestR for
// |dy| <= inner_thr in the same pass
int launch_hamming_knn2(const Geom &g, int n_pairs, const MatchParams &mp, bool train_sorted, const Buffers &b,
                        const uint32_t *counts, float inner_thr, cudaStream_t s);
// 512-bit rows (BRIEF-64, FREAK; match512.cu): desc64 = [n_images][kp_cap][64]; same keys and output arrays as the 256-bit kernels
int launch_hamming512_knn2(const Geom &g, int n_pairs, const MatchParams &mp, const uint8_t *desc64, const Buffers &b,
                           const uint32_t *counts, cudaStream_t s);
int launch_hamming512_cross(const Geom &g, int n_pairs, const uint8_t *desc64, const Buffers &b, const uint32_t *counts, cudaStream_t s);
// float descriptors (b.fdesc, 128-float rows; dim = 64 or 128), keys (float bits of d^2 << 32 | index)
int launch_l2_match(const Geom &g, int n_pairs, int dim, const MatchParams &mp, bool masked, bool all, const Buffers &b,
                    const uint32_t *counts, cudaStream_t s);
int launch_l2_band(const Geom &g, int n_pairs, int dim, const MatchParams &mp, const Buffers &b, const uint32_t *counts,
                   cudaStream_t s);
int launch_l2_tensor(const Geom &g, int n_pairs, int dim, bool need_second, const Buffers &b, const uint32_t *counts,
                     int phase, cudaStream_t s);
// exact cross-check + |dy| <= max_dy by band candidates + ONE tcgen05 GEMM + verification (l2verify.cu)
int launch_l2_band_cand(const Geom &g, int n_pairs, int dim, const MatchParams &mp, float inner, bool write_knn, const Buffers &b,
                        const uint32_t *counts, cudaStream_t s);
int launch_l2_verify(const Geom &g, int n_pairs, int dim, const Buffers &b, const uint32_t *counts, int phase, cudaStream_t s);
size_t l2_verify_list_entries(int kp_cap);
int launch_l2_finalize_ratio(const Geom &g, int n_pairs, double ratio, const Buffers &b, const uint32_t *counts, cudaStream_t s);
int launch_l2_finalize_cross(const Geom &g, int n_pairs, float max_dy, const Buffers &b, const uint32_t *counts, cudaStream_t s);
// liveGraph on float rows: the 64-bit-key twin of launch_finalize_cross_both
int launch_l2_finalize_cross_both(const Geom &g, int n_pairs, const uint32_t *counts, const unsigned long long *abL,
                                  const unsigned long long *cbL, const unsigned long long *abR, const unsigned long long *cbR,
                                  fe_match *out, uint32_t *n_out, cudaStream_t s);
int launch_finalize_ratio(const Geom &g, int n_pairs, double ratio, const Buffers &b,
                          const uint32_t *counts, cudaStream_t s);
int launch_finalize_cross(const Geom &g, int n_pairs, float max_dy, const Buffers &b,
                          const uint32_t *counts, cudaStream_t s);
// liveGraph: mutual matches of the left descriptors AND of the right descriptors with the same partner (algorithm.py:1160-1190)
int launch_finalize_cross_both(const Geom &g, int n_pairs, const uint32_t *counts, const uint32_t *abL, const uint32_t *cbL,
                               const uint32_t *abR, const uint32_t *cbR, fe_match *out, uint32_t *n_out, cudaStream_t s);

}  // namespace fe
