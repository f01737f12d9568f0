// Brute-force Hamming matching on 256-bit descriptors: LOP3 (xor / carry-save) + POPC on 32-bit
// words, with the reference's mask predicates evaluated in-register instead of materialising an
// Nq x Nt mask.
//
// Replaces:
//   * the O(N^2) host mask loops  /root/reference src/StereoCamera.cpp:182-196 (epipolar band),
//     src/front_end/algorithm.py:825-836, src/WindowMatcher.cpp:104-128 (search box);
//   * BFMatcher::knnMatch(q, t, k=2, mask)   StereoCamera.cpp:199-201, WindowMatcher.cpp:150-153,
//     algorithm.py:848-853      -> (best, second) per query among mask-allowed trains;
//   * BFMatcher(crossCheck=true)::match      src/live_stereo.cpp:240,364, features.py:670,724
//     -> unmasked row arg-min (allbest) and column arg-min (colbest).
// Keys are (distance << 16 | index): an unsigned min yields the smallest distance and, among ties,
// the lowest index -- OpenCV's stable ordering (SURVEY.md A.5).  Requires index < 65536.
//
// Four kernels:
//   hamming_cross_kernel  all Nq x Nt pairs, no mask (OpenCV asserts mask.empty() with crossCheck).
//                         A CTA owns THREADS*QPT queries in registers and streams the train
//                         descriptors through shared memory; every train word is a warp-wide
//                         broadcast LDS.128 amortised over QPT queries per lane.  POPC issues on
//                         the 16-lane XU pipe and bounds the kernel, so three of the eight xor
//                         words are first folded by carry-save adders (LOP3 0x96 / 0xE8 on the
//                         64-lane ALU pipe): 5 POPCs per 256-bit distance instead of 8.
//   hamming_band_tile_kernel  epipolar-masked kNN-2 when the train keypoints are in raster order
//                         (always true for keypoints this library detected): the allowed trains of a
//                         query are one contiguous index range read from a row table, so only ~1 %
//                         of the pairs are evaluated.  One thread per query; a CTA stages the trains
//                         its 256 queries need in shared memory.
//   hamming_band_kernel   the same for the window mask (WindowMatcher), one warp per query.
//   hamming_match_kernel  masked kNN-2 over all pairs, for caller-supplied keypoints in any order.
#include <algorithm>
#include <cstdlib>

#include "fe_internal.cuh"

namespace fe {

constexpr int TT = 256;   // train descriptors per shared-memory tile

template <int MASK>
__device__ __forceinline__ bool allowed(float qx, float qy, float tx, float ty, const MatchParams &mp) {
    if (MASK == FE_MASK_EPIPOLAR) return fabsf(__fsub_rn(qy, ty)) <= mp.epi_threshold;
    if (MASK == FE_MASK_WINDOW)
        return fabsf(__fsub_rn(qx, tx)) < mp.half_w && fabsf(__fsub_rn(qy, ty)) < mp.half_h;
    return true;
}

__device__ __forceinline__ uint32_t xor3(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}
__device__ __forceinline__ uint32_t maj3(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0xE8;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}

__device__ __forceinline__ uint32_t mad16(uint32_t d, uint32_t idx) {
    uint32_t r;
    asm("mad.lo.u32 %0, %1, 65536, %2;" : "=r"(r) : "r"(d), "r"(idx));
    return r;
}

// cv::NORM_HAMMING2 (ORB with WTA_K = 3 / 4, src/StereoCamera.cpp:504-511): the descriptor is 128 two-bit symbols and
// the distance counts differing SYMBOLS -- fold each bit pair of the xor word onto its low bit before counting.
template <bool H2>
__device__ __forceinline__ uint32_t xdiff(uint32_t a, uint32_t b) {
    const uint32_t x = a ^ b;
    return H2 ? ((x | (x >> 1)) & 0x55555555u) : x;
}

// popcount(q ^ t) over 256 bits with 5 POPCs: three 3:2 carry-save compressors first.
template <bool H2 = false>
__device__ __forceinline__ uint32_t hamming256_csa(const uint32_t (&q)[8], const uint4 &ta, const uint4 &tb) {
    const uint32_t x0 = xdiff<H2>(q[0], ta.x), x1 = xdiff<H2>(q[1], ta.y), x2 = xdiff<H2>(q[2], ta.z), x3 = xdiff<H2>(q[3], ta.w);
    const uint32_t x4 = xdiff<H2>(q[4], tb.x), x5 = xdiff<H2>(q[5], tb.y), x6 = xdiff<H2>(q[6], tb.z), x7 = xdiff<H2>(q[7], tb.w);
    const uint32_t s0 = xor3(x0, x1, x2), c0 = maj3(x0, x1, x2);
    const uint32_t s1 = xor3(x3, x4, x5), c1 = maj3(x3, x4, x5);
    const uint32_t s2 = xor3(s0, s1, x6), c2 = maj3(s0, s1, x6);
    const uint32_t ones = __popc(s2) + __popc(x7);
    const uint32_t twos = __popc(c0) + __popc(c1) + __popc(c2);
    return ones + 2u * twos;
}

template <bool H2 = false>
__device__ __forceinline__ uint32_t hamming256(const uint32_t (&q)[8], const uint4 &ta, const uint4 &tb) {
    return __popc(xdiff<H2>(q[0], ta.x)) + __popc(xdiff<H2>(q[1], ta.y)) + __popc(xdiff<H2>(q[2], ta.z)) +
           __popc(xdiff<H2>(q[3], ta.w)) + __popc(xdiff<H2>(q[4], tb.x)) + __popc(xdiff<H2>(q[5], tb.y)) +
           __popc(xdiff<H2>(q[6], tb.z)) + __popc(xdiff<H2>(q[7], tb.w));
}

// ---- unmasked row / column arg-min (cross-check) -------------------------------------------------
template <int QPT, int THREADS, bool H2 = false>
__global__ void __launch_bounds__(THREADS)
hamming_cross_kernel(Geom g, const uint32_t *__restrict__ counts, const uint8_t *__restrict__ desc,
                     uint32_t *__restrict__ allbest_out, uint32_t *__restrict__ colbest) {
    __shared__ uint4 s_desc[TT * 2];
    __shared__ uint32_t s_col[TT];

    const int pair = blockIdx.y;
    const int qi = 2 * pair, ti = 2 * pair + 1;
    const int nq = min((int)counts[qi], g.kp_cap), nt = min((int)counts[ti], g.kp_cap);
    const int q0 = blockIdx.x * (THREADS * QPT);
    if (q0 >= nq) return;
    const int lane = threadIdx.x & 31;

    uint32_t q[QPT][8];
    uint32_t allb[QPT], qkey[QPT];
#pragma unroll
    for (int j = 0; j < QPT; ++j) {
        // queries of one lane are THREADS apart so that a warp's loads stay coalesced
        const int qidx = q0 + j * THREADS + threadIdx.x;
        const bool valid = qidx < nq;
        const int src = valid ? qidx : nq - 1;
        const uint4 *p = reinterpret_cast<const uint4 *>(desc + ((size_t)qi * g.kp_cap + src) * 32);
        const uint4 a = __ldg(p), b = __ldg(p + 1);
        q[j][0] = a.x; q[j][1] = a.y; q[j][2] = a.z; q[j][3] = a.w;
        q[j][4] = b.x; q[j][5] = b.y; q[j][6] = b.z; q[j][7] = b.w;
        allb[j] = KEY_NONE;
        // an out-of-range lane re-evaluates the last query; its column key can never win a tie
        // against the real one (same distance, index 0xFFFF) and its row result is not stored
        qkey[j] = valid ? (uint32_t)qidx : 0xFFFFu;
    }

    const uint4 *tdesc = reinterpret_cast<const uint4 *>(desc + (size_t)ti * g.kp_cap * 32);
    uint32_t *col = colbest + (size_t)pair * g.kp_cap;

    for (int t0 = 0; t0 < nt; t0 += TT) {
        const int tn = min(TT, nt - t0);
        __syncthreads();
        for (int i = threadIdx.x; i < tn * 2; i += THREADS) s_desc[i] = __ldg(tdesc + (size_t)t0 * 2 + i);
        for (int i = threadIdx.x; i < tn; i += THREADS) s_col[i] = KEY_NONE;
        __syncthreads();
#pragma unroll 2
        for (int t = 0; t < tn; ++t) {
            const uint4 ta = s_desc[2 * t], tb = s_desc[2 * t + 1];
            const uint32_t tidx = (uint32_t)(t0 + t);
            uint32_t cmin = KEY_NONE;
#pragma unroll
            for (int j = 0; j < QPT; ++j) {
                // key = distance * 65536 + index as one IMAD each (FMA pipe) instead of shift + OR (ALU pipe,
                // which the xor / carry-save LOP3s already load as heavily as the POPCs load the XU pipe)
                const uint32_t d = hamming256_csa<H2>(q[j], ta, tb);
                allb[j] = min(allb[j], mad16(d, tidx));
                cmin = min(cmin, mad16(d, qkey[j]));
            }
            cmin = __reduce_min_sync(0xffffffffu, cmin);
            if (lane == 0) atomicMin(&s_col[t], cmin);
        }
        __syncthreads();
        for (int i = threadIdx.x; i < tn; i += THREADS) atomicMin(&col[t0 + i], s_col[i]);
    }
#pragma unroll
    for (int j = 0; j < QPT; ++j)
        if (qkey[j] != 0xFFFFu) allbest_out[(size_t)pair * g.kp_cap + qkey[j]] = allb[j];
}

// ---- banded kNN-2 for raster-ordered train keypoints ---------------------------------------------
// First index in [0, n) for which pred is true (pred is monotone false -> true), n if none.
// All 32 lanes cooperate: 32 probes per round.
template <typename Pred>
__device__ __forceinline__ int warp_first_true(int n, int lane, Pred pred) {
    int lo = 0, hi = n;                 // answer in [lo, hi]
    while (hi > lo) {
        const int span = hi - lo;
        const int step = (span + 31) >> 5;
        const int p = lo + lane * step;
        const bool v = p < hi ? pred(p) : true;
        const uint32_t m = __ballot_sync(0xffffffffu, v);
        const int f = m ? __ffs(m) - 1 : 32;   // first probing lane that sees true; 32: beyond lane 31's probe
        // probes f-1 (false) and f (true, or past hi) bracket the answer
        const int new_hi = min(lo + f * step, hi);
        const int new_lo = f == 0 ? lo : lo + (f - 1) * step + 1;
        if (f == 0) return lo;
        lo = new_lo; hi = new_hi;
    }
    return lo;
}

constexpr int BAND_WARPS = 8;
constexpr int BAND_LIST = 256;           // per-warp candidate list of the window-mask variant

// rowstart[image][r] = first keypoint index with floor(y) >= r (y non-decreasing); thread t fills the rows that start at t
__global__ void rowstart_kernel(Geom g, const uint32_t *__restrict__ counts, const float *__restrict__ ky, int *__restrict__ rowstart) {
    const int image = blockIdx.y, h = g.rs_h;
    const int n = min((int)counts[image], g.kp_cap);
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    int *rows = rowstart + (size_t)image * (h + 2);
    if (n == 0) {
        if (blockIdx.x == 0) for (int r = threadIdx.x; r <= h + 1; r += blockDim.x) rows[r] = 0;
        return;
    }
    if (t >= n) return;
    const float *y = ky + (size_t)image * g.kp_cap;
    const int rt = min(max((int)floorf(y[t]), 0), h);
    const int rp = t == 0 ? -1 : min(max((int)floorf(y[t - 1]), 0), h);
    for (int r = rp + 1; r <= rt; ++r) rows[r] = t;
    if (t == n - 1) for (int r = rt + 1; r <= h + 1; ++r) rows[r] = n;
}

int launch_rowstart(const Geom &g, const Buffers &b, const uint32_t *counts, cudaStream_t s) {
    rowstart_kernel<<<dim3(div_up(g.kp_cap, 256), g.n_images), 256, 0, s>>>(g, counts, b.ky, b.rowstart);
    return 1;
}

// ---- epipolar band, one thread per query over shared-memory train chunks --------------------------------------------------
// The band of a query holds ~36 trains at the bench's densities, about one per lane of a warp: a warp per query spent its time
// on the dependent round trips (row table, two ballot trims, scattered train rows, a global atomic per inner-band pair), not on
// the distances.  Here a CTA takes BT_Q consecutive query indices, one per thread, and stages the span of train rows its
// queries need -- [min lo, max hi) of their row-table ranges, ~290 trains for a block of detected keypoints -- in shared memory
// with coalesced loads.  Each thread walks its own range over the staged rows (lanes of one image row read the same train at
// the same step: broadcasts) and applies band_trim's exact predicate itself; y is non-decreasing, so that keeps the same run.
// Keys are unique (they carry the index), so best / second / inner best do not depend on the visiting order.
// Optional inner band (col_out != nullptr): pairs with |yq - yt| <= inner_thr also feed the cross-check's band candidates --
// row arg-min to inner_best, column arg-min to col_out (the band is symmetric, so this pass sees every pair of every train's
// band).  The column keys meet in shared memory and leave with one global atomicMin per staged train: the trains at a block's
// edge are shared with the neighbouring CTAs.
constexpr int BT_Q = 256;      // queries per CTA, one per thread
constexpr int BT_T = 512;      // trains per chunk: 16 KB of rows, 2 KB of y, 2 KB of column keys (a bench block's span fits one)

template <bool H2>
__global__ void __launch_bounds__(BT_Q, 4)
hamming_band_tile_kernel(Geom g, MatchParams mp, const uint32_t *__restrict__ counts, const uint8_t *__restrict__ desc,
                         const float *__restrict__ ky, uint32_t *__restrict__ best_out, uint32_t *__restrict__ second_out,
                         float inner_thr, uint32_t *__restrict__ inner_best, uint32_t *__restrict__ col_out,
                         const int *__restrict__ rowstart) {
    __shared__ uint4 s_desc[BT_T * 2];
    __shared__ float s_ty[BT_T];
    __shared__ uint32_t s_col[BT_T];
    __shared__ int s_lo, s_hi;
    const int pair = blockIdx.y;
    const int qi = 2 * pair, ti = 2 * pair + 1;
    const int nq = min((int)counts[qi], g.kp_cap), nt = min((int)counts[ti], g.kp_cap);
    if ((int)blockIdx.x * BT_Q >= nq) return;
    const int qidx = blockIdx.x * BT_Q + threadIdx.x;
    const bool valid = qidx < nq;
    const float reach = mp.epi_threshold;
    float qy = 0.f;
    int lo = nt, hi = 0;                 // empty unless the thread has a query
    uint32_t q[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (valid) {
        qy = __fadd_rn(ky[(size_t)qi * g.kp_cap + qidx], mp.q_off);
        band_range(rowstart + (size_t)ti * (g.rs_h + 2), g.rs_h, qy - mp.t_off, reach, lo, hi);
        hi = min(hi, nt);
        const uint4 *p = reinterpret_cast<const uint4 *>(desc + ((size_t)qi * g.kp_cap + qidx) * 32);
        const uint4 a = __ldg(p), b = __ldg(p + 1);
        q[0] = a.x; q[1] = a.y; q[2] = a.z; q[3] = a.w; q[4] = b.x; q[5] = b.y; q[6] = b.z; q[7] = b.w;
    }
    // the CTA's span: min lo / max hi over all its threads -- queries may come in any order
    if (threadIdx.x == 0) { s_lo = nt; s_hi = 0; }
    __syncthreads();
    const int wlo = __reduce_min_sync(0xffffffffu, lo < hi ? lo : nt), whi = __reduce_max_sync(0xffffffffu, lo < hi ? hi : 0);
    if ((threadIdx.x & 31) == 0) { atomicMin(&s_lo, wlo); atomicMax(&s_hi, whi); }
    __syncthreads();
    const int span_lo = s_lo, span_hi = s_hi;

    const uint4 *tdesc = reinterpret_cast<const uint4 *>(desc + (size_t)ti * g.kp_cap * 32);
    const float *tky = ky + (size_t)ti * g.kp_cap;
    uint32_t *col = col_out ? col_out + (size_t)pair * g.kp_cap : nullptr;
    uint32_t best = KEY_NONE, second = KEY_NONE, ibest = KEY_NONE;
    for (int c0 = span_lo; c0 < span_hi; c0 += BT_T) {
        const int cn = min(BT_T, span_hi - c0);
        __syncthreads();                 // the previous chunk is measured and flushed
        for (int i = threadIdx.x; i < 2 * cn; i += BT_Q) s_desc[i] = __ldg(tdesc + 2 * (size_t)c0 + i);
        for (int i = threadIdx.x; i < cn; i += BT_Q) {
            s_ty[i] = tky[c0 + i];
            if (col) s_col[i] = KEY_NONE;
        }
        __syncthreads();
        const int e = min(hi, c0 + cn);
        for (int t = max(lo, c0); t < e; ++t) {
            const int k = t - c0;
            const float ty = s_ty[k];
            const float d = __fsub_rn(qy, __fadd_rn(ty, mp.t_off));
            if (d <= reach && !(d < -reach)) {
                const uint32_t d16 = hamming256<H2>(q, s_desc[2 * k], s_desc[2 * k + 1]) << 16;
                const uint32_t key = d16 | (uint32_t)t;
                second = min(second, max(best, key));
                best = min(best, key);
                if (col && fabsf(__fsub_rn(qy, ty)) <= inner_thr) {
                    ibest = min(ibest, key);
                    atomicMin(&s_col[k], d16 | (uint32_t)qidx);
                }
            }
        }
        if (col) {
            __syncthreads();
            for (int i = threadIdx.x; i < cn; i += BT_Q)
                if (s_col[i] != KEY_NONE) atomicMin(&col[c0 + i], s_col[i]);
        }
    }
    if (valid) {
        const size_t o = (size_t)pair * g.kp_cap + qidx;
        best_out[o] = best;
        second_out[o] = second;
        if (col) inner_best[o] = ibest;
    }
}

// ---- window-masked kNN-2 for raster-ordered train keypoints (WindowMatcher), one warp per query --------------------------
// (one CTA per SM minimum: the kernel carries its candidate list and more state and slows down when squeezed)
template <bool H2 = false>
__global__ void __launch_bounds__(BAND_WARPS * 32, 1)
hamming_band_kernel(Geom g, MatchParams mp, const uint32_t *__restrict__ counts,
                    const uint8_t *__restrict__ desc, const float *__restrict__ kx,
                    const float *__restrict__ ky, uint32_t *__restrict__ best_out,
                    uint32_t *__restrict__ second_out, const int *__restrict__ rowstart) {
    const int pair = blockIdx.y;
    const int qi = 2 * pair, ti = 2 * pair + 1;
    const int nq = min((int)counts[qi], g.kp_cap), nt = min((int)counts[ti], g.kp_cap);
    const int lane = threadIdx.x & 31;
    const int qidx = blockIdx.x * BAND_WARPS + (threadIdx.x >> 5);
    if (qidx >= nq) return;
    const float *tkx = kx + (size_t)ti * g.kp_cap, *tky = ky + (size_t)ti * g.kp_cap;
    const float qx = kx[(size_t)qi * g.kp_cap + qidx];
    const float qy = __fadd_rn(ky[(size_t)qi * g.kp_cap + qidx], mp.q_off);
    // candidate rows from the train image's row table (no search), trimmed to the exact allowed run with the float
    // arithmetic of allowed<FE_MASK_WINDOW>
    const float reach = mp.half_h;
    int lo, hi;
    band_range(rowstart + (size_t)ti * (g.rs_h + 2), g.rs_h, qy - mp.t_off, reach, lo, hi);
    hi = min(hi, nt);
    band_trim(lo, hi, lane, [&](int t) { return __fsub_rn(qy, __fadd_rn(tky[t], mp.t_off)) < reach; },
              [&](int t) { return __fsub_rn(qy, __fadd_rn(tky[t], mp.t_off)) <= -reach; });
    uint32_t q[8];
    {
        const uint4 *p = reinterpret_cast<const uint4 *>(desc + ((size_t)qi * g.kp_cap + qidx) * 32);
        const uint4 a = __ldg(p), b = __ldg(p + 1);
        q[0] = a.x; q[1] = a.y; q[2] = a.z; q[3] = a.w; q[4] = b.x; q[5] = b.y; q[6] = b.z; q[7] = b.w;
    }
    const uint4 *tdesc = reinterpret_cast<const uint4 *>(desc + (size_t)ti * g.kp_cap * 32);
    uint32_t best = KEY_NONE, second = KEY_NONE;
    auto measure = [&](int t) {
        const uint4 ta = __ldg(tdesc + 2 * (size_t)t), tb = __ldg(tdesc + 2 * (size_t)t + 1);
        const uint32_t key = (hamming256<H2>(q, ta, tb) << 16) | (uint32_t)t;
        second = min(second, max(best, key));
        best = min(best, key);
    };
    // The row range holds every keypoint of ~100 image rows; the |dx| test keeps ~8 % of them.  Testing and measuring in
    // the same loop would run the distance code in almost every round for two or three lanes: compact the survivors
    // into a per-warp list first (ballot + prefix), then measure them densely.
    __shared__ uint16_t s_list[BAND_WARPS][BAND_LIST];
    uint16_t *list = s_list[threadIdx.x >> 5];
    int cnt = 0;
    for (int t0 = lo; t0 < hi; t0 += 32) {
        const int t = t0 + lane;
        const bool pass = t < hi && fabsf(__fsub_rn(qx, tkx[t])) < mp.half_w;
        const uint32_t m = __ballot_sync(0xffffffffu, pass);
        if (pass) list[cnt + __popc(m & ((1u << lane) - 1u))] = (uint16_t)t;
        cnt += __popc(m);
        if (cnt > BAND_LIST - 32 || t0 + 32 >= hi) {
            __syncwarp();
#pragma unroll 1          // (unrolled, the kernel needs 72 registers instead of 40)
            for (int i = lane; i < cnt; i += 32) measure((int)list[i]);
            __syncwarp();
            cnt = 0;
        }
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) {
        const uint32_t ob = __shfl_xor_sync(0xffffffffu, best, off);
        const uint32_t os = __shfl_xor_sync(0xffffffffu, second, off);
        second = min(min(second, os), max(best, ob));
        best = min(best, ob);
    }
    if (lane == 0) {
        best_out[(size_t)pair * g.kp_cap + qidx] = best;
        second_out[(size_t)pair * g.kp_cap + qidx] = second;
    }
}

// ---- masked kNN-2 over all pairs (keypoints in any order) ----------------------------------------
template <int QPT, int THREADS, int MASK, bool H2 = false>
__global__ void __launch_bounds__(THREADS)
hamming_match_kernel(Geom g, MatchParams mp, const uint32_t *__restrict__ counts,
                     const uint8_t *__restrict__ desc, const float *__restrict__ kx,
                     const float *__restrict__ ky, uint32_t *__restrict__ best_out,
                     uint32_t *__restrict__ second_out) {
    __shared__ uint4 s_desc[TT * 2];
    __shared__ float s_tx[TT], s_ty[TT];

    const int pair = blockIdx.y;
    const int qi = 2 * pair, ti = 2 * pair + 1;
    const int nq = min((int)counts[qi], g.kp_cap), nt = min((int)counts[ti], g.kp_cap);
    const int q0 = blockIdx.x * (THREADS * QPT);
    if (q0 >= nq) return;

    uint32_t q[QPT][8];
    float qx[QPT], qy[QPT];
    uint32_t best[QPT], second[QPT];
    int qidx[QPT];
#pragma unroll
    for (int j = 0; j < QPT; ++j) {
        qidx[j] = q0 + j * THREADS + threadIdx.x;
        const int src = qidx[j] < nq ? qidx[j] : nq - 1;
        const uint4 *p = reinterpret_cast<const uint4 *>(desc + ((size_t)qi * g.kp_cap + src) * 32);
        const uint4 a = __ldg(p), b = __ldg(p + 1);
        q[j][0] = a.x; q[j][1] = a.y; q[j][2] = a.z; q[j][3] = a.w;
        q[j][4] = b.x; q[j][5] = b.y; q[j][6] = b.z; q[j][7] = b.w;
        qx[j] = kx[(size_t)qi * g.kp_cap + src];
        qy[j] = __fadd_rn(ky[(size_t)qi * g.kp_cap + src], mp.q_off);
        best[j] = second[j] = KEY_NONE;
    }

    const uint4 *tdesc = reinterpret_cast<const uint4 *>(desc + (size_t)ti * g.kp_cap * 32);
    const float *tkx = kx + (size_t)ti * g.kp_cap, *tky = ky + (size_t)ti * g.kp_cap;

    for (int t0 = 0; t0 < nt; t0 += TT) {
        const int tn = min(TT, nt - t0);
        __syncthreads();
        for (int i = threadIdx.x; i < tn * 2; i += THREADS) s_desc[i] = __ldg(tdesc + (size_t)t0 * 2 + i);
        for (int i = threadIdx.x; i < tn; i += THREADS) {
            s_tx[i] = tkx[t0 + i];
            s_ty[i] = __fadd_rn(tky[t0 + i], mp.t_off);
        }
        __syncthreads();
#pragma unroll 2
        for (int t = 0; t < tn; ++t) {
            const uint4 ta = s_desc[2 * t], tb = s_desc[2 * t + 1];
            const float tx = s_tx[t], ty = s_ty[t];
            const uint32_t tidx = (uint32_t)(t0 + t);
#pragma unroll
            for (int j = 0; j < QPT; ++j) {
                const uint32_t key = (hamming256_csa<H2>(q[j], ta, tb) << 16) | tidx;
                if (allowed<MASK>(qx[j], qy[j], tx, ty, mp)) {
                    second[j] = min(second[j], max(best[j], key));
                    best[j] = min(best[j], key);
                }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < QPT; ++j) {
        if (qidx[j] >= nq) continue;
        const size_t o = (size_t)pair * g.kp_cap + qidx[j];
        best_out[o] = best[j];
        second_out[o] = second[j];
    }
}

// ---- POPC-pipe throughput probe (roofline denominator of the matcher; bench.py) ------------------
__global__ void __launch_bounds__(256) popc_peak_kernel(int iters, uint32_t seed, uint32_t *sink) {
    uint32_t x[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = seed * (threadIdx.x + 1u) + 0x9E3779B9u * (i + 1u);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] = __popc(x[i]) | 0x55550000u;    // 8 independent POPC chains; the OR shares an ALU slot
    }
    uint32_t acc = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) acc += x[i];
    if (acc == 0xDEADBEEFu) sink[0] = acc;      // never true; keeps the chains alive
}

double launch_popc_peak(int sms, int iters, uint32_t *sink, cudaStream_t s) {
    const int ctas = sms * 8;
    popc_peak_kernel<<<ctas, 256, 0, s>>>(iters, 12345u, sink);
    return (double)ctas * 256.0 * 8.0 * iters;
}

int launch_hamming_cross(const Geom &g, int n_pairs, bool h2, const Buffers &b, const uint32_t *counts, cudaStream_t s) {
    cudaMemsetAsync(b.colbest, 0xFF, sizeof(uint32_t) * (size_t)n_pairs * g.kp_cap, s);
    if (h2) {      // NORM_HAMMING2: same kernels, symbol-wise distance
        if (n_pairs >= 4) { dim3 grid(div_up(g.kp_cap, 256), n_pairs); hamming_cross_kernel<2, 128, true><<<grid, 128, 0, s>>>(g, counts, b.desc, b.allbest, b.colbest); }
        else { dim3 grid(div_up(g.kp_cap, 64), n_pairs); hamming_cross_kernel<1, 64, true><<<grid, 64, 0, s>>>(g, counts, b.desc, b.allbest, b.colbest); }
        return 1;
    }
    // 256-query CTAs (2 per lane, 128 threads) keep the per-pair remainder small and won the launch-shape
    // sweep on B200; a lone pair would leave most of the 148 SMs idle, so it gets 64-query CTAs.
    static const int variant = getenv("FE_CROSS_VARIANT") ? atoi(getenv("FE_CROSS_VARIANT")) : 0;   // tuning sweeps only
#define FE_CROSS_GO(Q, T) { dim3 grid(div_up(g.kp_cap, Q * T), n_pairs); \
                            hamming_cross_kernel<Q, T><<<grid, T, 0, s>>>(g, counts, b.desc, b.allbest, b.colbest); }
    if (n_pairs >= 4) {
        switch (variant) {
        case 1: FE_CROSS_GO(4, 128); break;
        case 8: FE_CROSS_GO(3, 128); break;
        case 14: FE_CROSS_GO(4, 64); break;
        default: FE_CROSS_GO(2, 128); break;     // best of the sweep (gpurun_out/sweep_cross*.log): 4.05 ms vs 4.42 ms for <4, 64>
        }
    } else {
        dim3 grid(div_up(g.kp_cap, 64), n_pairs);
        hamming_cross_kernel<1, 64><<<grid, 64, 0, s>>>(g, counts, b.desc, b.allbest, b.colbest);
    }
    return 1;
}

int launch_hamming_knn2(const Geom &g, int n_pairs, const MatchParams &mp, bool train_sorted, const Buffers &b,
                        const uint32_t *counts, float inner_thr, cudaStream_t s) {
    if (train_sorted && mp.mask != FE_MASK_NONE) {
        if (inner_thr >= 0.f) cudaMemsetAsync(b.cx_bestR, 0xFF, sizeof(uint32_t) * (size_t)n_pairs * g.kp_cap, s);
        launch_rowstart(g, b, counts, s);
        if (mp.mask == FE_MASK_EPIPOLAR) {
            dim3 grid(div_up(g.kp_cap, BT_Q), n_pairs);
#define FE_BAND_GO(H2) hamming_band_tile_kernel<H2><<<grid, BT_Q, 0, s>>>(g, mp, counts, b.desc, b.ky, b.best, b.second, inner_thr, \
            inner_thr >= 0.f ? b.cx_bestL : nullptr, inner_thr >= 0.f ? b.cx_bestR : nullptr, b.rowstart)
            if (mp.h2) FE_BAND_GO(true); else FE_BAND_GO(false);
#undef FE_BAND_GO
        } else {
            dim3 grid(div_up(g.kp_cap, BAND_WARPS), n_pairs);
#define FE_BAND_GO(H2) hamming_band_kernel<H2><<<grid, BAND_WARPS * 32, 0, s>>>(g, mp, counts, b.desc, b.kx, b.ky, b.best, b.second, b.rowstart)
            if (mp.h2) FE_BAND_GO(true); else FE_BAND_GO(false);
#undef FE_BAND_GO
        }
        return 2;
    }
    if (mp.h2) {
#define FE_MATCH_GO2(MASK) hamming_match_kernel<1, 64, MASK, true><<<dim3(div_up(g.kp_cap, 64), n_pairs), 64, 0, s>>>( \
        g, mp, counts, b.desc, b.kx, b.ky, b.best, b.second)
        if (mp.mask == FE_MASK_EPIPOLAR) FE_MATCH_GO2(FE_MASK_EPIPOLAR);
        else if (mp.mask == FE_MASK_WINDOW) FE_MATCH_GO2(FE_MASK_WINDOW);
        else FE_MATCH_GO2(FE_MASK_NONE);
#undef FE_MATCH_GO2
        return 1;
    }
#define FE_MATCH_GO(QPT, THREADS, MASK)                                                             \
    hamming_match_kernel<QPT, THREADS, MASK><<<dim3(div_up(g.kp_cap, QPT * THREADS), n_pairs), THREADS, 0, s>>>( \
        g, mp, counts, b.desc, b.kx, b.ky, b.best, b.second)
    if (n_pairs >= 4) {
        if (mp.mask == FE_MASK_EPIPOLAR) FE_MATCH_GO(4, 64, FE_MASK_EPIPOLAR);
        else if (mp.mask == FE_MASK_WINDOW) FE_MATCH_GO(4, 64, FE_MASK_WINDOW);
        else FE_MATCH_GO(4, 64, FE_MASK_NONE);
    } else {
        if (mp.mask == FE_MASK_EPIPOLAR) FE_MATCH_GO(1, 64, FE_MASK_EPIPOLAR);
        else if (mp.mask == FE_MASK_WINDOW) FE_MATCH_GO(1, 64, FE_MASK_WINDOW);
        else FE_MATCH_GO(1, 64, FE_MASK_NONE);
    }
#undef FE_MATCH_GO
    return 1;
}

// ---- finalisation: Lowe ratio (mode A) and mutual check + |dy| filter (mode B) ----------------
constexpr int FIN_THREADS = 1024;


// Mode A: accept a row with one candidate, or with d0 < ratio*d1 (double arithmetic, strict) --
// StereoCamera.cpp:206-264, algorithm.py:838-846.  The C++ query-unique de-dup loop is a no-op
// because knnMatch returns one row per query.  Output ordered by queryIdx.
__device__ __forceinline__ void finalize_ratio_body(const Geom &g, double ratio, const uint32_t *__restrict__ counts,
                                                    const uint32_t *__restrict__ best, const uint32_t *__restrict__ second,
                                                    fe_match *__restrict__ out, uint32_t *__restrict__ n_out, uint32_t *s_warp) {
    const int pair = blockIdx.x;
    const int nq = min((int)counts[2 * pair], g.kp_cap);
    const uint32_t *b = best + (size_t)pair * g.kp_cap, *s2 = second + (size_t)pair * g.kp_cap;
    fe_match *o = out + (size_t)pair * g.kp_cap;
    uint32_t offset = 0;
    for (int base = 0; base < nq; base += FIN_THREADS) {
        const int i = base + threadIdx.x;
        bool good = false;
        uint32_t kb = KEY_NONE;
        if (i < nq) {
            kb = b[i];
            const uint32_t ks = s2[i];
            if (kb != KEY_NONE) {
                if (ks == KEY_NONE) good = true;
                else good = (double)(kb >> 16) < ratio * (double)(ks >> 16);
            }
        }
        uint32_t total;
        const uint32_t pos = offset + block_excl_scan_1024(good ? 1u : 0u, s_warp, total);
        if (good) {
            fe_match m;
            m.queryIdx = (uint32_t)i; m.trainIdx = kb & 0xFFFF; m.imgIdx = 0; m.distance = (float)(kb >> 16);
            o[pos] = m;
        }
        offset += total;
    }
    if (threadIdx.x == 0) n_out[pair] = offset;
}

__global__ void __launch_bounds__(FIN_THREADS)
finalize_ratio_kernel(Geom g, double ratio, const uint32_t *__restrict__ counts,
                      const uint32_t *__restrict__ best, const uint32_t *__restrict__ second,
                      fe_match *__restrict__ out, uint32_t *__restrict__ n_out) {
    __shared__ uint32_t s_warp[33];
    finalize_ratio_body(g, ratio, counts, best, second, out, n_out, s_warp);
}

// Mode B: keep (q, s) when s = argmin_t D[q,t], q = argmin_q' D[q',s] (first minima) and
// |yq - ys| <= max_dy -- live_stereo.cpp:364-377, features.py:724-733.  Ordered by queryIdx.
__global__ void __launch_bounds__(FIN_THREADS)
finalize_cross_kernel(Geom g, float max_dy, const uint32_t *__restrict__ counts,
                      const uint32_t *__restrict__ allbest, const uint32_t *__restrict__ colbest,
                      const float *__restrict__ ky, fe_match *__restrict__ out,
                      uint32_t *__restrict__ n_out) {
    __shared__ uint32_t s_warp[33];
    const int pair = blockIdx.x;
    const int nq = min((int)counts[2 * pair], g.kp_cap);
    const int nt = min((int)counts[2 * pair + 1], g.kp_cap);
    const uint32_t *ab = allbest + (size_t)pair * g.kp_cap, *cb = colbest + (size_t)pair * g.kp_cap;
    const float *qy = ky + (size_t)(2 * pair) * g.kp_cap, *ty = ky + (size_t)(2 * pair + 1) * g.kp_cap;
    fe_match *o = out + (size_t)pair * g.kp_cap;
    uint32_t offset = 0;
    for (int base = 0; base < nq; base += FIN_THREADS) {
        const int i = base + threadIdx.x;
        bool good = false;
        uint32_t kb = KEY_NONE;
        if (i < nq && nt > 0) {
            kb = ab[i];
            const uint32_t t = kb & 0xFFFF;
            good = (cb[t] & 0xFFFF) == (uint32_t)i;
            if (good && max_dy >= 0.f) good = fabsf(__fsub_rn(qy[i], ty[t])) <= max_dy;
        }
        uint32_t total;
        const uint32_t pos = offset + block_excl_scan_1024(good ? 1u : 0u, s_warp, total);
        if (good) {
            fe_match m;
            m.queryIdx = (uint32_t)i; m.trainIdx = kb & 0xFFFF; m.imgIdx = 0; m.distance = (float)(kb >> 16);
            o[pos] = m;
        }
        offset += total;
    }
    if (threadIdx.x == 0) n_out[pair] = offset;
}

// liveGraph's tracker (/root/reference src/front_end/algorithm.py:1160-1190): bf.match(crossCheck) of the current against
// the previous frame's LEFT descriptors and, separately, of the RIGHT descriptors; landmark c of the current frame
// continues landmark t of the previous one iff (c, t) is a mutual match on BOTH sides.  Ordered by c.
__global__ void __launch_bounds__(FIN_THREADS)
finalize_cross_both_kernel(Geom g, const uint32_t *__restrict__ counts, const uint32_t *__restrict__ abL,
                           const uint32_t *__restrict__ cbL, const uint32_t *__restrict__ abR, const uint32_t *__restrict__ cbR,
                           fe_match *__restrict__ out, uint32_t *__restrict__ n_out) {
    __shared__ uint32_t s_warp[33];
    const int pair = blockIdx.x;
    const int nq = min((int)counts[2 * pair], g.kp_cap), nt = min((int)counts[2 * pair + 1], g.kp_cap);
    const size_t o0 = (size_t)pair * g.kp_cap;
    fe_match *o = out + o0;
    uint32_t offset = 0;
    for (int base = 0; base < nq; base += FIN_THREADS) {
        const int i = base + threadIdx.x;
        bool good = false;
        uint32_t kl = KEY_NONE;
        if (i < nq && nt > 0) {
            kl = abL[o0 + i];
            const uint32_t kr = abR[o0 + i];
            const uint32_t tl = kl & 0xFFFF, tr = kr & 0xFFFF;
            good = tl == tr && (cbL[o0 + tl] & 0xFFFF) == (uint32_t)i && (cbR[o0 + tr] & 0xFFFF) == (uint32_t)i;
        }
        uint32_t total;
        const uint32_t pos = offset + block_excl_scan_1024(good ? 1u : 0u, s_warp, total);
        if (good) {
            fe_match m;
            m.queryIdx = (uint32_t)i; m.trainIdx = kl & 0xFFFF; m.imgIdx = 0; m.distance = (float)(kl >> 16);   // left distance
            o[pos] = m;
        }
        offset += total;
    }
    if (threadIdx.x == 0) n_out[pair] = offset;
}

int launch_finalize_cross_both(const Geom &g, int n_pairs, const uint32_t *counts, const uint32_t *abL, const uint32_t *cbL,
                               const uint32_t *abR, const uint32_t *cbR, fe_match *out, uint32_t *n_out, cudaStream_t s) {
    finalize_cross_both_kernel<<<n_pairs, FIN_THREADS, 0, s>>>(g, counts, abL, cbL, abR, cbR, out, n_out);
    return 1;
}

// ---- cross-check with candidate verification (exact, ~2x fewer instructions) ------------------------------------------
// The live nodes keep a cross-check match only if |yq - yt| <= max_dy (src/live_stereo.cpp:369-377, features.py:732-733).
// A surviving pair is therefore the BAND arg-min of its row and of its column, so the band passes (1 % of the pairs)
// name every possible survivor (q, t*, d*) -- what is left is to VERIFY that no train anywhere beats t* for q and no
// query anywhere beats q for t*.  A pair (q', t') can only do that if d(q', t') <= d*, and
//     LB(q', t') = popc( OR_w (q'_w ^ t'_w) )  <=  d(q', t')        (8 LOP3 "(a ^ b) | c" + ONE POPC)
// is a lower bound that sits at ~31.8 for unrelated descriptors (a bit position of the OR is clear only if all eight
// words agree there), while candidate distances are mostly <= 24.  So:
//   cross_classify_kernel   mutual band candidates, thresholds thr_q / thr_t (d* or -1), allbest / colbest seeded with the
//                           candidate keys, queries and trains partitioned into "easy" (d* <= 24 or no candidate) and "hard";
//   hamming_verify_kernel   <PRUNE = true>  easy x easy: LB first, the 256-bit distance only when some lane of the warp
//                                           has LB <= max(thr_q, thr_t) (1 % of the warp-iterations on the bench data);
//                           <PRUNE = false> hard queries x all trains, easy queries x hard trains: every distance;
//                           both fold what they evaluate into allbest / colbest with atomicMin on the usual keys, so ties
//                           resolve exactly as in the all-pairs kernel (skipped pairs have d > d* and cannot win or tie);
//   finalize_cross_cand_kernel  a candidate survives iff its keys are still the row and column minima.
// Results are identical to hamming_cross_kernel + finalize_cross_kernel (tests compare against cv2 and the oracle).
//
// Multi-index join (exact) for the bulk of the work.  Fifteen or fewer differing bits spread over the sixteen 16-bit halves
// of a descriptor leave at least one half IDENTICAL (pigeonhole).  So an entry whose threshold is <= 15 (class A, ~92 %) can
// only be disturbed by a partner that shares a half with it:
//   mih_transpose_kernel   halves of every entry in permutation order ([image][half position][k], coalesced for the join) and
//                          the index of its own mutual candidate (already seeded, never re-measured);
//   mih_join_kernel<0>     one CTA per (pair, half position): the class-A trains' halves go into a shared-memory hash table,
//                          every class-A query looks up its own half and measures the few trains it finds -- chance
//                          collisions, ~0.1 per probe, which leave after the distance.  (R = 1 also probes the 16 one-bit
//                          neighbours -- valid up to 31 differing bits; measured slower than the LB scan for class B.)
// The LB scan then only serves class B (15 < d* <= CX_T, ~5 %) against A + B, and class C (d* > CX_T, ~3 %) is evaluated
// in full against everything.  Without the join (per-image capacity above MIH_MAX) class A is empty and the LB scan serves
// B x B as before.
// 128-bit rows (BRIEF-16) ride zero-padded in the 256-bit rows: their halves 8 .. 15 are 0 for every entry, so a join at those
// positions would put every class-A train into one probe run and measure every pair.  The join then covers the 8 data halves
// only, and class A ends at 7 differing bits -- the pigeonhole of 8 halves.  The LB4 / LB8 scans stay valid on the zero words.
constexpr int CX_T = 24;             // B / C split of the LB scan (the LB4 filter stops paying above it)
constexpr int CX_T2 = 48;            // C / D split: the two-POPC LB8 filter serves thresholds up to here, class D is evaluated in full

__global__ void __launch_bounds__(1024)
cross_classify_kernel(Geom g, int t1, int t2, int t3, const uint32_t *__restrict__ counts, const uint32_t *__restrict__ bestL,
                      const uint32_t *__restrict__ bestR, const uint32_t *__restrict__ wide_best,
                      uint32_t *__restrict__ allbest, uint32_t *__restrict__ colbest,
                      int *__restrict__ thrq, int *__restrict__ thrt, uint16_t *__restrict__ qperm,
                      uint16_t *__restrict__ tperm, uint32_t *__restrict__ cxn) {
    __shared__ uint32_t s_warp[33];
    const int pair = blockIdx.x;
    const size_t o = (size_t)pair * g.kp_cap;
    {
        const int side = blockIdx.y;       // one CTA per (pair, side): the kernel is all latency (block scans), more CTAs = more SMs busy
        const int n = min((int)counts[2 * pair + side], g.kp_cap);
        const uint32_t *mine = (side ? bestR : bestL) + o, *other = (side ? bestL : bestR) + o;
        uint32_t *seed = (side ? colbest : allbest) + o;
        int *thr = (side ? thrt : thrq) + o;
        uint16_t *perm = (side ? tperm : qperm) + o;
        // pass 1: validity, thresholds, seeds, class A (d* <= t1, or no candidate) to the front of the permutation
        uint32_t n_cls[4] = {0, 0, 0, 0};
        for (int base = 0; base < n; base += 1024) {
            const int i = base + threadIdx.x;
            bool mine_now = false;
            if (i < n) {
                const uint32_t key = mine[i];
                bool valid = key != KEY_NONE && (other[key & 0xFFFF] & 0xFFFF) == (uint32_t)i;
                // wide_best (mode A's kNN-2 over the wider epipolar band, same launch): a query whose best key there is
                // smaller than its inner-band candidate's has a closer train outside the inner band -- the candidate is not
                // its row minimum, so the PAIR is dead for both sides (kills ~2/3 of the false candidates, d* ~ 100)
                if (valid && wide_best) {
                    const uint32_t q = side ? (key & 0xFFFF) : (uint32_t)i;
                    valid = wide_best[o + q] == bestL[o + q];
                }
                const int d = valid ? (int)(key >> 16) : -1;
                seed[i] = valid ? key : KEY_NONE;
                thr[i] = d;
                mine_now = d <= t1;
            }
            uint32_t total;
            const uint32_t pos = block_excl_scan_1024(mine_now ? 1u : 0u, s_warp, total);
            if (mine_now) perm[n_cls[0] + pos] = (uint16_t)i;
            n_cls[0] += total;
        }
        // passes 2 - 4: class B (t1 < d* <= t2), class C (t2 < d* <= t3), class D (d* > t3)
        for (int cls = 1; cls < 4; ++cls) {
            uint32_t first = n_cls[0] + (cls >= 2 ? n_cls[1] : 0u) + (cls >= 3 ? n_cls[2] : 0u);
            for (int base = 0; base < n; base += 1024) {
                const int i = base + threadIdx.x;
                const int d = i < n ? thr[i] : -1;
                const bool mine_now = i < n && (cls == 1 ? (d > t1 && d <= t2) : cls == 2 ? (d > t2 && d <= t3) : d > t3);
                uint32_t total;
                const uint32_t pos = block_excl_scan_1024(mine_now ? 1u : 0u, s_warp, total);
                if (mine_now) perm[first + n_cls[cls] + pos] = (uint16_t)i;
                n_cls[cls] += total;
            }
        }
        if (threadIdx.x == 0) { cxn[8 * pair + 4 * side] = n_cls[0]; cxn[8 * pair + 4 * side + 1] = n_cls[1]; cxn[8 * pair + 4 * side + 2] = n_cls[2]; cxn[8 * pair + 4 * side + 3] = n_cls[3]; }
    }
}

__device__ __forceinline__ int class_prefix(const uint32_t *n, int c) {       // entries in classes [0, c)
    return (int)((c > 0 ? n[0] : 0u) + (c > 1 ? n[1] : 0u) + (c > 2 ? n[2] : 0u) + (c > 3 ? n[3] : 0u));
}

__device__ __forceinline__ uint32_t or_xor(uint32_t a, uint32_t b, uint32_t c) {      // (a ^ b) | c
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0xBE;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}

// region = qc0 | qc1 << 4 | tc0 << 8 | tc1 << 12: query classes [qc0, qc1) x train classes [tc0, tc1) of the permutations
// (A = 0, B = 1, C = 2).  PRUNE is only valid when every threshold of the region is <= CX_T (no class C on either side).
// blockIdx.z splits the region's train list into gridDim.z contiguous chunks (row results meet in allbest by atomicMin),
// so that the few hard queries of region 1 still spread over the whole GPU.
// The prefilter uses the first four words only: LB4 = popc((q0^t0)|(q1^t1)|(q2^t2)|(q3^t3)) <= d.  Against the exact
// per-pair threshold max(thr_q, thr_t) (candidate distances are ~8 on average) it lets ~3 % of the warp-iterations through.
// PRUNE = 2: LB8 = LB4 + the same bound on words 4 .. 7 (two POPCs, sits near 59 for unrelated descriptors: 0.03 % of the
// pairs fall under a threshold of 40, 0.7 % under 48) -- serves class C (CX_T < d* <= CX_T2) at about half the
// instructions of the full distance.
template <int PRUNE, int VQ, int VTHREADS>
__global__ void __launch_bounds__(VTHREADS)
hamming_verify_kernel(Geom g, int region, const uint32_t *__restrict__ cxn, const uint8_t *__restrict__ desc,
                      const uint16_t *__restrict__ qperm, const uint16_t *__restrict__ tperm,
                      const int *__restrict__ thrq, const int *__restrict__ thrt, uint32_t *__restrict__ allbest,
                      uint32_t *__restrict__ colbest) {
    __shared__ uint4 s_desc[TT * 2];
    __shared__ uint32_t s_col[TT];
    __shared__ int s_thr[TT];
    __shared__ uint16_t s_idx[TT];
    const int pair = blockIdx.y;
    const size_t o = (size_t)pair * g.kp_cap;
    // bit 16 of `region`: the two sides trade places -- lanes own TRAINS (classes in bits 0 .. 7), the tiles hold QUERIES (bits
    // 8 .. 15).  Row and column minima are symmetric (keys distance << 16 | the other side's index, atomicMin), so this is a
    // swap of pointers; it lets a region with a few hundred queries and thousands of trains run with full warps and one tile.
    const bool swapped = (region >> 16) & 1;
    if (swapped) {
        const uint16_t *tp = qperm; qperm = tperm; tperm = tp;
        const int *tt = thrq; thrq = thrt; thrt = tt;
        uint32_t *tb = allbest; allbest = colbest; colbest = tb;
    }
    const uint32_t *nq_cls = cxn + 8 * pair + (swapped ? 4 : 0), *nt_cls = cxn + 8 * pair + (swapped ? 0 : 4);
    const int q_first = class_prefix(nq_cls, region & 15), q_count = class_prefix(nq_cls, (region >> 4) & 15) - q_first;
    const int t_first = class_prefix(nt_cls, (region >> 8) & 15), t_all = class_prefix(nt_cls, (region >> 12) & 15) - t_first;
    const int chunk = round_up(div_up(t_all, (int)gridDim.z), TT);
    const int t_begin = blockIdx.z * chunk, t_end = min(t_all, t_begin + chunk);
    if (t_begin >= t_end) return;
    const int lane = threadIdx.x & 31;
    const uint8_t *qdesc = desc + (size_t)(2 * pair + (swapped ? 1 : 0)) * g.kp_cap * 32, *tdesc = desc + (size_t)(2 * pair + (swapped ? 0 : 1)) * g.kp_cap * 32;

    // query blocks of this CTA: gridDim.x may be smaller than the region needs (the few-query regions are launched with one
    // or two CTAs per train chunk instead of cap / (VQ * VTHREADS) CTAs that would all but one exit at once: an empty CTA
    // still costs ~0.25 us of launch throughput per 1000, which was 0.1 ms per step for the class-C / D passes)
    for (int q0 = blockIdx.x * (VTHREADS * VQ); q0 < q_count; q0 += gridDim.x * (VTHREADS * VQ)) {
    uint32_t q[VQ][8], allb[VQ], qkey[VQ];
    int qthr[VQ];
#pragma unroll
    for (int j = 0; j < VQ; ++j) {
        const int k = q0 + j * VTHREADS + threadIdx.x;
        const bool valid = k < q_count;
        const int qi = (int)qperm[o + q_first + (valid ? k : q_count - 1)];
        const uint4 *p = reinterpret_cast<const uint4 *>(qdesc + (size_t)qi * 32);
        const uint4 a = __ldg(p), b = __ldg(p + 1);
        q[j][0] = a.x; q[j][1] = a.y; q[j][2] = a.z; q[j][3] = a.w;
        q[j][4] = b.x; q[j][5] = b.y; q[j][6] = b.z; q[j][7] = b.w;
        allb[j] = KEY_NONE;
        // a padding lane repeats the last query: same distances, but its column key carries index 0xFFFF and so can never
        // win a tie against the real one; its row result is not stored
        qkey[j] = valid ? (uint32_t)qi : 0xFFFFu;
        qthr[j] = valid ? thrq[o + qi] : -1;
    }
    for (int t0 = t_begin; t0 < t_end; t0 += TT) {
        const int tn = min(TT, t_end - t0);
        __syncthreads();
        for (int i = threadIdx.x; i < tn; i += VTHREADS) {
            const int ti = (int)tperm[o + t_first + t0 + i];
            const uint4 *p = reinterpret_cast<const uint4 *>(tdesc + (size_t)ti * 32);
            s_desc[2 * i] = __ldg(p); s_desc[2 * i + 1] = __ldg(p + 1);
            s_idx[i] = (uint16_t)ti;
            s_thr[i] = thrt[o + ti];
            s_col[i] = KEY_NONE;
        }
        __syncthreads();
#pragma unroll 2
        for (int t = 0; t < tn; ++t) {
            const uint4 ta = s_desc[2 * t];
            if (PRUNE == 1) {
                const int tthr = s_thr[t];
                bool need = false;
                int lbmin = 64;
#pragma unroll
                for (int j = 0; j < VQ; ++j) {
                    uint32_t acc = q[j][0] ^ ta.x;
                    acc = or_xor(q[j][1], ta.y, acc); acc = or_xor(q[j][2], ta.z, acc); acc = or_xor(q[j][3], ta.w, acc);
                    const int lb = (int)__popc(acc);
                    need = need || lb <= qthr[j];
                    lbmin = min(lbmin, lb);
                }
                need = need || lbmin <= tthr;
                if (!__any_sync(0xffffffffu, need)) continue;
            }
            const uint4 tb = s_desc[2 * t + 1];
            if (PRUNE == 2) {
                const int tthr = s_thr[t];
                bool need = false;
                int lbmin = 64;
#pragma unroll
                for (int j = 0; j < VQ; ++j) {
                    uint32_t a0 = q[j][0] ^ ta.x, a1 = q[j][4] ^ tb.x;
                    a0 = or_xor(q[j][1], ta.y, a0); a0 = or_xor(q[j][2], ta.z, a0); a0 = or_xor(q[j][3], ta.w, a0);
                    a1 = or_xor(q[j][5], tb.y, a1); a1 = or_xor(q[j][6], tb.z, a1); a1 = or_xor(q[j][7], tb.w, a1);
                    const int lb = (int)(__popc(a0) + __popc(a1));
                    need = need || lb <= qthr[j];
                    lbmin = min(lbmin, lb);
                }
                need = need || lbmin <= tthr;
                if (!__any_sync(0xffffffffu, need)) continue;
            }
            const uint32_t tidx = (uint32_t)s_idx[t];
            uint32_t cmin = KEY_NONE;
#pragma unroll
            for (int j = 0; j < VQ; ++j) {
                const uint32_t d = hamming256_csa(q[j], ta, tb);
                allb[j] = min(allb[j], mad16(d, tidx));
                cmin = min(cmin, mad16(d, qkey[j]));
            }
            cmin = __reduce_min_sync(0xffffffffu, cmin);
            if (lane == 0) atomicMin(&s_col[t], cmin);
        }
        __syncthreads();
        for (int i = threadIdx.x; i < tn; i += VTHREADS)
            if (s_col[i] != KEY_NONE) atomicMin(&colbest[o + s_idx[i]], s_col[i]);
    }
#pragma unroll
    for (int j = 0; j < VQ; ++j)
        if (qkey[j] != 0xFFFFu && allb[j] != KEY_NONE) atomicMin(&allbest[o + qkey[j]], allb[j]);
    }
}

// Halves in permutation order + own-candidate index, for every entry of every image of the batch (see above).
__global__ void __launch_bounds__(256)
mih_transpose_kernel(Geom g, const uint32_t *__restrict__ counts, const uint8_t *__restrict__ desc,
                     const uint16_t *__restrict__ qperm, const uint16_t *__restrict__ tperm,
                     const uint32_t *__restrict__ bestL, const uint32_t *__restrict__ bestR,
                     const int *__restrict__ thrq, const int *__restrict__ thrt, uint16_t *__restrict__ half,
                     uint16_t *__restrict__ star) {
    const int image = blockIdx.y, pair = image >> 1, side = image & 1;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= min((int)counts[image], g.kp_cap)) return;
    const size_t o = (size_t)pair * g.kp_cap;
    const uint32_t idx = (side ? tperm : qperm)[o + k];
    const uint4 *p = reinterpret_cast<const uint4 *>(desc + ((size_t)image * g.kp_cap + idx) * 32);
    const uint4 a = __ldg(p), b = __ldg(p + 1);
    const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    uint16_t *h = half + (size_t)image * 16 * g.kp_cap + k;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        h[(size_t)(2 * i) * g.kp_cap] = (uint16_t)(w[i] & 0xFFFFu);
        h[(size_t)(2 * i + 1) * g.kp_cap] = (uint16_t)(w[i] >> 16);
    }
    const bool has = (side ? thrt : thrq)[o + idx] >= 0;
    star[(size_t)image * g.kp_cap + k] = has ? (uint16_t)((side ? bestR : bestL)[o + idx] & 0xFFFFu) : (uint16_t)0xFFFFu;
}

__device__ __forceinline__ uint32_t mih_hash(uint32_t half, uint32_t mask) { return ((half * 40503u) >> 1) & mask; }

// spec = table side (0 queries / 1 trains) | table classes [c0, c1) << 4, << 8 | probe classes [c0, c1) << 12, << 16.
// Shared memory: open-addressing hash table (linear probing, load factor <= 1/2) of the table side's entries keyed by their
// 16-bit half at position blockIdx.x; an entry is (half << 16 | descriptor index).  Equal halves sit in one probe run.
template <int R>
__global__ void __launch_bounds__(1024, 2)
mih_join_kernel(Geom g, int slots, int spec, int dmax, const uint32_t *__restrict__ cxn, const uint8_t *__restrict__ desc,
                const uint16_t *__restrict__ qperm, const uint16_t *__restrict__ tperm, const uint16_t *__restrict__ half,
                const uint16_t *__restrict__ star, uint32_t *__restrict__ allbest, uint32_t *__restrict__ colbest) {
    extern __shared__ uint32_t s_tab[];
    const int pos16 = blockIdx.x, pair = blockIdx.y;
    const size_t o = (size_t)pair * g.kp_cap;
    const int tside = spec & 1, pside = tside ^ 1;
    const uint32_t *nT = cxn + 8 * pair + 4 * tside, *nP = cxn + 8 * pair + 4 * pside;
    const int t_first = class_prefix(nT, (spec >> 4) & 15), nt = class_prefix(nT, (spec >> 8) & 15) - t_first;
    const int p_first = class_prefix(nP, (spec >> 12) & 15), np = class_prefix(nP, (spec >> 16) & 15) - p_first;
    if (np == 0 || nt == 0) return;
    const int timg = 2 * pair + tside, pimg = 2 * pair + pside;
    const uint8_t *tdesc = desc + (size_t)timg * g.kp_cap * 32, *pdesc = desc + (size_t)pimg * g.kp_cap * 32;
    const uint16_t *tperm_ = (tside ? tperm : qperm) + o, *pperm_ = (pside ? tperm : qperm) + o;
    const uint16_t *thalf = half + ((size_t)timg * 16 + pos16) * g.kp_cap, *phalf = half + ((size_t)pimg * 16 + pos16) * g.kp_cap;
    const uint16_t *pstar = star + (size_t)pimg * g.kp_cap;
    int S = 64;
    while (S < 2 * nt) S <<= 1;
    S = min(S, slots);                             // host sized the allocation for 2 * kp_cap
    const uint32_t mask = (uint32_t)S - 1u;
    for (int i = threadIdx.x; i < S; i += 1024) s_tab[i] = KEY_NONE;
    __syncthreads();
    for (int i = threadIdx.x; i < nt; i += 1024) {
        const uint32_t hv = thalf[t_first + i];
        const uint32_t key = (hv << 16) | (uint32_t)tperm_[t_first + i];
        uint32_t slot = mih_hash(hv, mask);
        while (atomicCAS(&s_tab[slot], KEY_NONE, key) != KEY_NONE) slot = (slot + 1) & mask;
    }
    __syncthreads();
    for (int k = threadIdx.x; k < np; k += 1024) {
        const uint32_t hv = phalf[p_first + k];
        const uint32_t pidx = pperm_[p_first + k], own = pstar[p_first + k];
        uint32_t q[8];
        bool loaded = false;
#pragma unroll 1
        for (int v = 0; v < (R ? 17 : 1); ++v) {
            const uint32_t want = v == 0 ? hv : hv ^ (1u << (v - 1));
            uint32_t slot = mih_hash(want, mask);
            for (uint32_t key = s_tab[slot]; key != KEY_NONE; slot = (slot + 1) & mask, key = s_tab[slot]) {
                if ((key >> 16) != want) continue;
                const uint32_t tidx = key & 0xFFFFu;
                if (tidx == own) continue;          // the entry's own mutual candidate: already seeded by the classify kernel
                if (!loaded) {
                    const uint4 *qp = reinterpret_cast<const uint4 *>(pdesc + (size_t)pidx * 32);
                    const uint4 qa = __ldg(qp), qb = __ldg(qp + 1);
                    q[0] = qa.x; q[1] = qa.y; q[2] = qa.z; q[3] = qa.w; q[4] = qb.x; q[5] = qb.y; q[6] = qb.z; q[7] = qb.w;
                    loaded = true;
                }
                const uint4 *tp = reinterpret_cast<const uint4 *>(tdesc + (size_t)tidx * 32);
                const uint4 ta = __ldg(tp), tb = __ldg(tp + 1);
                // chance collisions (d ~ 128) leave here; a close pair is found at every half it shares, atomicMin is idempotent
                const uint32_t d = hamming256_csa(q, ta, tb);
                if (d > (uint32_t)dmax) continue;   // cannot disturb a pair whose thresholds are both <= dmax
                const uint32_t qi = tside ? pidx : tidx, ti = tside ? tidx : pidx;
                atomicMin(&allbest[o + qi], mad16(d, ti));
                atomicMin(&colbest[o + ti], mad16(d, qi));
            }
        }
    }
}

__device__ __forceinline__ void finalize_cross_cand_body(const Geom &g, const uint32_t *__restrict__ counts, const uint32_t *__restrict__ bestL,
                                                         const uint32_t *__restrict__ bestR, const int *__restrict__ thrq,
                                                         const uint32_t *__restrict__ allbest, const uint32_t *__restrict__ colbest,
                                                         fe_match *__restrict__ out, uint32_t *__restrict__ n_out, uint32_t *s_warp) {
    const int pair = blockIdx.x;
    const size_t o0 = (size_t)pair * g.kp_cap;
    const int nq = min((int)counts[2 * pair], g.kp_cap);
    fe_match *o = out + o0;
    uint32_t offset = 0;
    for (int base = 0; base < nq; base += FIN_THREADS) {
        const int i = base + threadIdx.x;
        bool good = false;
        uint32_t kb = KEY_NONE;
        if (i < nq && thrq[o0 + i] >= 0) {
            kb = bestL[o0 + i];
            const uint32_t t = kb & 0xFFFF;
            good = allbest[o0 + i] == kb && colbest[o0 + t] == bestR[o0 + t];     // still the row and the column minimum
        }
        uint32_t total;
        const uint32_t pos = offset + block_excl_scan_1024(good ? 1u : 0u, s_warp, total);
        if (good) {
            fe_match m;
            m.queryIdx = (uint32_t)i; m.trainIdx = kb & 0xFFFF; m.imgIdx = 0; m.distance = (float)(kb >> 16);
            o[pos] = m;
        }
        offset += total;
    }
    if (threadIdx.x == 0) n_out[pair] = offset;
}

__global__ void __launch_bounds__(FIN_THREADS)
finalize_cross_cand_kernel(Geom g, const uint32_t *__restrict__ counts, const uint32_t *__restrict__ bestL,
                           const uint32_t *__restrict__ bestR, const int *__restrict__ thrq,
                           const uint32_t *__restrict__ allbest, const uint32_t *__restrict__ colbest,
                           fe_match *__restrict__ out, uint32_t *__restrict__ n_out) {
    __shared__ uint32_t s_warp[33];
    finalize_cross_cand_body(g, counts, bestL, bestR, thrq, allbest, colbest, out, n_out, s_warp);
}

// Mode A's ratio test and mode B's candidate check in ONE launch (blockIdx.y picks the mode): both are one 1024-thread CTA per
// pair that is all latency (six block scans), so two launches of n_pairs CTAs each leave most SMs idle twice.
__global__ void __launch_bounds__(FIN_THREADS)
finalize_cand_and_ratio_kernel(Geom g, const uint32_t *__restrict__ counts, const uint32_t *__restrict__ bestL,
                               const uint32_t *__restrict__ bestR, const int *__restrict__ thrq,
                               const uint32_t *__restrict__ allbest, const uint32_t *__restrict__ colbest,
                               fe_match *__restrict__ out_b, uint32_t *__restrict__ n_b, double ratio,
                               const uint32_t *__restrict__ best, const uint32_t *__restrict__ second,
                               fe_match *__restrict__ out_a, uint32_t *__restrict__ n_a) {
    __shared__ uint32_t s_warp[33];
    if (blockIdx.y == 0) finalize_cross_cand_body(g, counts, bestL, bestR, thrq, allbest, colbest, out_b, n_b, s_warp);
    else finalize_ratio_body(g, ratio, counts, best, second, out_a, n_a, s_warp);
}

// cross-check + |dy| <= max_dy for raster-ordered keypoints on both sides; writes match_b / n_b
int launch_hamming_cross_pruned(const Geom &g, int n_pairs, float max_dy, bool have_band, bool use_join, int row_bytes, const Buffers &b,
                                const uint32_t *counts, double fused_ratio, cudaStream_t s, cudaStream_t aux, cudaEvent_t ev_fork,
                                cudaEvent_t ev_join) {
    MatchParams mp{};
    mp.mask = FE_MASK_EPIPOLAR; mp.epi_threshold = max_dy;
    if (!have_band) {      // (otherwise mode A's band pass already produced cx_bestL / cx_bestR as its inner band)
        cudaMemsetAsync(b.cx_bestR, 0xFF, sizeof(uint32_t) * (size_t)n_pairs * g.kp_cap, s);
        launch_rowstart(g, b, counts, s);
        hamming_band_tile_kernel<false><<<dim3(div_up(g.kp_cap, BT_Q), n_pairs), BT_Q, 0, s>>>(
            g, mp, counts, b.desc, b.ky, reinterpret_cast<uint32_t *>(b.cx_thrq) /* scratch until classify */, b.cx_dummy, max_dy,
            b.cx_bestL, b.cx_bestR, b.rowstart);
    }
    const bool mih = use_join && g.kp_cap <= MIH_MAX && b.cx_half;
    // A / B split: the join's positions are the rows' 16-bit halves, and at most halves - 1 differing bits leave one identical
    const int halves = row_bytes / 2, join_t1 = halves - 1;
    // without the join class A is empty (t1 = -2: even "no candidate" entries, d* = -1, fall into class B)
    static const int cx_t = getenv("FE_CX_T") ? atoi(getenv("FE_CX_T")) : CX_T;      // B / C split (tuning knob; any value is exact)
    static const int cx_t2 = std::max(cx_t, getenv("FE_CX_T2") ? atoi(getenv("FE_CX_T2")) : CX_T2);   // C / D split (likewise)
    static const bool wide_kill = !(getenv("FE_CX_WIDE") && atoi(getenv("FE_CX_WIDE")) == 0);        // A/B testing
    // the splits must not decrease: a B / C split below the A / B split would put an entry into class A and class D at once
    const int t1 = mih ? join_t1 : -2, t2 = std::max(cx_t, t1), t3 = std::max(cx_t2, t2);
    cross_classify_kernel<<<dim3(n_pairs, 2), 1024, 0, s>>>(g, t1, t2, t3, counts, b.cx_bestL, b.cx_bestR,
                                                   have_band && wide_kill ? b.best : nullptr, b.allbest,
                                                   b.colbest, b.cx_thrq, b.cx_thrt, b.cx_qperm, b.cx_tperm, b.cx_n);
    int n_launch = have_band ? 5 : 6;
#define FE_JOIN_SPEC(tside, tc0, tc1, pc0, pc1) ((tside) | (tc0) << 4 | (tc1) << 8 | (pc0) << 12 | (pc1) << 16)
    // transpose + join only read what classify wrote and fold their findings with atomicMin, like the verification scans: they
    // may run beside them (side stream forked after classify, joined before finalize)
    cudaStream_t js = s;
    if (mih && aux) { cudaEventRecord(ev_fork, s); cudaStreamWaitEvent(aux, ev_fork, 0); js = aux; }
    if (mih) {
        mih_transpose_kernel<<<dim3(div_up(g.kp_cap, 256), 2 * n_pairs), 256, 0, js>>>(g, counts, b.desc, b.cx_qperm, b.cx_tperm, b.cx_bestL, b.cx_bestR,
                                                                                      b.cx_thrq, b.cx_thrt, b.cx_half, b.cx_star);
        int S = 64;
        while (S < 2 * g.kp_cap) S <<= 1;
        const size_t smem = sizeof(uint32_t) * (size_t)S;
        if (smem > 48 * 1024) {
            cudaFuncSetAttribute(mih_join_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        }
#define FE_JOIN_ARGS b.cx_n, b.desc, b.cx_qperm, b.cx_tperm, b.cx_half, b.cx_star, b.allbest, b.colbest
        mih_join_kernel<0><<<dim3(halves, n_pairs), 1024, smem, js>>>(g, S, FE_JOIN_SPEC(1, 0, 1, 0, 1), join_t1, FE_JOIN_ARGS);   // A trains | A queries
        if (js != s) cudaEventRecord(ev_join, js);
#undef FE_JOIN_ARGS
        n_launch += 3;
    }
#undef FE_JOIN_SPEC
    static const int vvar = getenv("FE_VERIFY_VARIANT") ? atoi(getenv("FE_VERIFY_VARIANT")) : 0;     // tuning sweeps only
#define FE_VERIFY_ARGS g, b.cx_n, b.desc, b.cx_qperm, b.cx_tperm, b.cx_thrq, b.cx_thrt, b.allbest, b.colbest
    // X = 0: one CTA per query block of the whole capacity (regions with thousands of queries); X > 0: that many CTAs per
    // (pair, train chunk), looping over the region's query blocks (regions with a few hundred queries at most)
#define FE_VERIFY_GO(PR, Q, T, REGION, Z, X) hamming_verify_kernel<PR, Q, T><<<dim3((X) ? (X) : div_up(g.kp_cap, Q * T), n_pairs, Z), T, 0, s>>>( \
        g, REGION, b.cx_n, b.desc, b.cx_qperm, b.cx_tperm, b.cx_thrq, b.cx_thrt, b.allbest, b.colbest)
    const int few = n_pairs >= 8 ? 1 : 4;
#define FE_REGION(qc0, qc1, tc0, tc1) ((qc0) | (qc1) << 4 | (tc0) << 8 | (tc1) << 12)
#define FE_SWAPPED (1 << 16)
    if (mih) {
        // launch shapes from a sweep on B200 (24 train chunks keep ~50 warps per SM busy for the ~220 class-B queries)
        static const bool swap_b = !(getenv("FE_CX_SWAP") && atoi(getenv("FE_CX_SWAP")) == 0);
        if (swap_b) FE_VERIFY_GO(1, 2, 128, FE_SWAPPED | FE_REGION(0, 2, 1, 2), 1, 0);      // (A + B) trains x B queries, LB scan
        else FE_VERIFY_GO(1, 2, 128, FE_REGION(1, 2, 0, 2), 24, few);     // B queries x (A + B) trains, LB scan
        FE_VERIFY_GO(1, 2, 128, FE_REGION(0, 1, 1, 2), 1, 0);      // A queries x B trains, LB scan
    } else {
        const int r0 = FE_REGION(0, 2, 0, 2);                      // (A is empty) B x B, LB scan
        switch (vvar) {
        case 1: FE_VERIFY_GO(1, 4, 64, r0, 2, 0); break;
        case 2: FE_VERIFY_GO(1, 8, 64, r0, 4, 0); break;
        case 3: FE_VERIFY_GO(1, 2, 128, r0, 2, 0); break;
        case 4: FE_VERIFY_GO(1, 8, 128, r0, 4, 0); break;
        default: FE_VERIFY_GO(1, 4, 128, r0, 4, 0); break;
        }
    }
    static const int zc = getenv("FE_CX_ZC") ? atoi(getenv("FE_CX_ZC")) : 24, zd = getenv("FE_CX_ZD") ? atoi(getenv("FE_CX_ZD")) : 32;   // tuning sweeps only
    static const bool swap_few = !(getenv("FE_CX_SWAP") && atoi(getenv("FE_CX_SWAP")) == 0);                                                // A/B testing
    if (swap_few) {
        // few queries x many trains: lanes own the trains, the queries are the tile (one CTA per 256 trains, no train chunks)
        FE_VERIFY_GO(2, 2, 128, FE_SWAPPED | FE_REGION(0, 3, 2, 3), 1, 0);    // (A + B + C) trains x class-C queries, LB8 scan
        FE_VERIFY_GO(2, 2, 128, FE_REGION(0, 2, 2, 3), 1, 0);                 // A + B queries x class-C trains, LB8 scan
        FE_VERIFY_GO(0, 2, 128, FE_SWAPPED | FE_REGION(0, 4, 3, 4), 1, 0);    // every train x the few class-D queries, in full
        FE_VERIFY_GO(0, 2, 128, FE_REGION(0, 3, 3, 4), 1, 0);                 // A + B + C queries x the few class-D trains, in full
    } else {
        FE_VERIFY_GO(2, 1, 128, FE_REGION(2, 3, 0, 3), zc, few);          // the ~100 class-C queries x (A + B + C) trains, LB8 scan
        FE_VERIFY_GO(2, 2, 128, FE_REGION(0, 2, 2, 3), 1, 0);           // A + B queries x class-C trains, LB8 scan
        FE_VERIFY_GO(0, 1, 64, FE_REGION(3, 4, 0, 4), zd, few);           // the few class-D queries x every train, in full
        FE_VERIFY_GO(0, 2, 128, FE_REGION(0, 3, 3, 4), 1, 0);           // A + B + C queries x the few class-D trains, in full
    }
    n_launch += 2;
#undef FE_REGION
#undef FE_SWAPPED
#undef FE_VERIFY_GO
#undef FE_VERIFY_ARGS
    if (js != s) cudaStreamWaitEvent(s, ev_join, 0);
    if (fused_ratio >= 0.0)      // mode A's finalize rides along (its kNN-2 pass ran before this stage)
        finalize_cand_and_ratio_kernel<<<dim3(n_pairs, 2), FIN_THREADS, 0, s>>>(g, counts, b.cx_bestL, b.cx_bestR, b.cx_thrq, b.allbest, b.colbest,
                                                                                b.match_b, b.n_b, fused_ratio, b.best, b.second, b.match_a, b.n_a);
    else
        finalize_cross_cand_kernel<<<n_pairs, FIN_THREADS, 0, s>>>(g, counts, b.cx_bestL, b.cx_bestR, b.cx_thrq, b.allbest, b.colbest,
                                                                  b.match_b, b.n_b);
    return n_launch;
}

int launch_finalize_ratio(const Geom &g, int n_pairs, double ratio, const Buffers &b,
                          const uint32_t *counts, cudaStream_t s) {
    finalize_ratio_kernel<<<n_pairs, FIN_THREADS, 0, s>>>(g, ratio, counts, b.best, b.second,
                                                          b.match_a, b.n_a);
    return 1;
}

int launch_finalize_cross(const Geom &g, int n_pairs, float max_dy, const Buffers &b,
                          const uint32_t *counts, cudaStream_t s) {
    finalize_cross_kernel<<<n_pairs, FIN_THREADS, 0, s>>>(g, max_dy, counts, b.allbest, b.colbest,
                                                          b.ky, b.match_b, b.n_b);
    return 1;
}

}  // namespace fe
