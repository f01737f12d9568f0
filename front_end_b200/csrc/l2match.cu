// Brute-force L2 matching of float descriptors (SURF 64-d / SURF_EXTENDED 128-d), exact FP32 form.
//
// Replaces BFMatcher(NORM_L2)::knnMatch(q, t, 2, mask) and BFMatcher(NORM_L2, crossCheck)::match for
// the reference's float descriptors (getMatcher, /root/reference src/front_end/features.py:463-467;
// StereoCamera.cpp:199-201 with normType L2; algorithm.py:848-853), with the same mask predicates as
// the Hamming path evaluated in-register.
//
// d^2 = sum_k (q_k - t_k)^2 is accumulated directly (no |q|^2 + |t|^2 - 2 q.t cancellation), k
// ascending, one FADD + one FFMA per term.  Keys are 64-bit (float bits of d^2 << 32 | index): d^2 >= 0,
// so unsigned order == numeric order and ties resolve to the lowest index (OpenCV's stable order).
// The reported distance is sqrtf(d^2), as cv::batchDistance does for NORM_L2.
//
// Tiling: a CTA owns 64 queries (shared memory, k-major) and streams 64-train tiles; 16 x 16 threads,
// 4 x 4 register micro-tile each.  Row results (masked best / second, unmasked best) are merged
// across the 16 threads of a row with half-warp shuffles; column minima (cross-check) go through
// shared then global 64-bit atomicMin.
#include "fe_internal.cuh"
#include <type_traits>

namespace fe {

constexpr int LT = 64;            // queries per CTA == trains per tile
constexpr int LPAD = LT + 4;      // k-major row pitch (floats): keeps float4 alignment, spreads banks
constexpr unsigned long long KEY64_NONE = 0xFFFFFFFFFFFFFFFFull;

template <int MASK>
__device__ __forceinline__ bool allowed_f(float qx, float qy, float tx, float ty, const MatchParams &mp) {
    if (MASK == FE_MASK_EPIPOLAR) return fabsf(__fsub_rn(qy, ty)) <= mp.epi_threshold;
    if (MASK == FE_MASK_WINDOW)
        return fabsf(__fsub_rn(qx, tx)) < mp.half_w && fabsf(__fsub_rn(qy, ty)) < mp.half_h;
    return true;
}

__device__ __forceinline__ void push2(unsigned long long &best, unsigned long long &second, unsigned long long key) {
    second = min(second, max(best, key));
    best = min(best, key);
}

template <int D, int MASK, bool WANT_MASKED, bool WANT_ALL>
__global__ void __launch_bounds__(256)
l2_match_kernel(Geom g, MatchParams mp, const uint32_t *__restrict__ counts, const float *__restrict__ fdesc,
                const float *__restrict__ kx, const float *__restrict__ ky, unsigned long long *__restrict__ best_out,
                unsigned long long *__restrict__ second_out, unsigned long long *__restrict__ allbest_out,
                unsigned long long *__restrict__ colbest) {
    extern __shared__ __align__(16) float smem[];
    float *s_q = smem;                      // [D][LPAD]
    float *s_t = smem + D * LPAD;           // [D][LPAD]
    __shared__ float s_tx[LT], s_ty[LT];
    __shared__ unsigned long long s_col[LT];

    const int pair = blockIdx.y;
    const int qi = 2 * pair, ti = 2 * pair + 1;
    const int nq = min((int)counts[qi], g.kp_cap), nt = min((int)counts[ti], g.kp_cap);
    const int q0 = blockIdx.x * LT;
    if (q0 >= nq) return;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const float *qd = fdesc + ((size_t)qi * g.kp_cap + q0) * 128;
    const float *td = fdesc + (size_t)ti * g.kp_cap * 128;

    // queries -> shared, k-major; rows past nq repeat the last valid query (never stored)
    for (int i = tid; i < LT * (D / 4); i += 256) {
        const int r = i / (D / 4), c4 = i - r * (D / 4);
        const int rr = min(r, nq - 1 - q0);
        const float4 v = *reinterpret_cast<const float4 *>(qd + (size_t)rr * 128 + 4 * c4);
        s_q[(4 * c4 + 0) * LPAD + r] = v.x; s_q[(4 * c4 + 1) * LPAD + r] = v.y;
        s_q[(4 * c4 + 2) * LPAD + r] = v.z; s_q[(4 * c4 + 3) * LPAD + r] = v.w;
    }
    float qx[4], qy[4];
    unsigned long long best[4], second[4], allb[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const int q = min(q0 + ty * 4 + a, nq - 1);
        qx[a] = kx[(size_t)qi * g.kp_cap + q];
        qy[a] = __fadd_rn(ky[(size_t)qi * g.kp_cap + q], mp.q_off);
        best[a] = second[a] = allb[a] = KEY64_NONE;
    }
    const float *tkx = kx + (size_t)ti * g.kp_cap, *tky = ky + (size_t)ti * g.kp_cap;
    unsigned long long *col = colbest + (size_t)pair * g.kp_cap;

    for (int t0 = 0; t0 < nt; t0 += LT) {
        const int tn = min(LT, nt - t0);
        __syncthreads();
        for (int i = tid; i < LT * (D / 4); i += 256) {
            const int r = i / (D / 4), c4 = i - r * (D / 4);
            const int rr = min(r, tn - 1);
            const float4 v = *reinterpret_cast<const float4 *>(td + (size_t)(t0 + rr) * 128 + 4 * c4);
            s_t[(4 * c4 + 0) * LPAD + r] = v.x; s_t[(4 * c4 + 1) * LPAD + r] = v.y;
            s_t[(4 * c4 + 2) * LPAD + r] = v.z; s_t[(4 * c4 + 3) * LPAD + r] = v.w;
        }
        if (tid < LT) {
            const int rr = min(tid, tn - 1);
            s_tx[tid] = tkx[t0 + rr];
            s_ty[tid] = __fadd_rn(tky[t0 + rr], mp.t_off);
            s_col[tid] = KEY64_NONE;
        }
        __syncthreads();
        float acc[4][4];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
#pragma unroll 8
        for (int k = 0; k < D; ++k) {
            const float4 qa = *reinterpret_cast<const float4 *>(s_q + k * LPAD + ty * 4);
            const float4 tb = *reinterpret_cast<const float4 *>(s_t + k * LPAD + tx * 4);
            const float qv[4] = {qa.x, qa.y, qa.z, qa.w}, tv[4] = {tb.x, tb.y, tb.z, tb.w};
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    const float df = __fsub_rn(qv[a], tv[b]);
                    acc[a][b] = __fmaf_rn(df, df, acc[a][b]);
                }
        }
        unsigned long long cmin[4] = {KEY64_NONE, KEY64_NONE, KEY64_NONE, KEY64_NONE};
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int tl = tx * 4 + b;
            if (tl >= tn) continue;
            const float txx = s_tx[tl], tyy = s_ty[tl];
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                const unsigned long long bits = (unsigned long long)__float_as_uint(acc[a][b]) << 32;
                const unsigned long long key = bits | (unsigned)(t0 + tl);
                if (WANT_MASKED && allowed_f<MASK>(qx[a], qy[a], txx, tyy, mp)) push2(best[a], second[a], key);
                if (WANT_ALL) {
                    allb[a] = min(allb[a], key);
                    const int q = q0 + ty * 4 + a;
                    if (q < nq) cmin[b] = min(cmin[b], bits | (unsigned)q);
                }
            }
        }
        if (WANT_ALL) {
#pragma unroll
            for (int b = 0; b < 4; ++b)
                if (cmin[b] != KEY64_NONE) atomicMin(&s_col[tx * 4 + b], cmin[b]);
            __syncthreads();
            if (tid < tn) atomicMin(&col[t0 + tid], s_col[tid]);
        }
    }
    // merge the 16 threads (tx = 0..15, one half-warp) that share a query row
#pragma unroll
    for (int a = 0; a < 4; ++a) {
#pragma unroll
        for (int off = 8; off; off >>= 1) {
            if (WANT_MASKED) {
                const unsigned long long ob = __shfl_xor_sync(0xffffffffu, best[a], off);
                const unsigned long long os = __shfl_xor_sync(0xffffffffu, second[a], off);
                second[a] = min(min(second[a], os), max(best[a], ob));
                best[a] = min(best[a], ob);
            }
            if (WANT_ALL) allb[a] = min(allb[a], __shfl_xor_sync(0xffffffffu, allb[a], off));
        }
        const int q = q0 + ty * 4 + a;
        if (tx == 0 && q < nq) {
            const size_t o = (size_t)pair * g.kp_cap + q;
            if (WANT_MASKED) { best_out[o] = best[a]; second_out[o] = second[a]; }
            if (WANT_ALL) allbest_out[o] = allb[a];
        }
    }
}

// ---- banded kNN-2 for raster-ordered train keypoints (the L2 twin of hamming_band_kernel) -----------------
template <typename Pred>
__device__ __forceinline__ int warp_first_true_f(int n, int lane, Pred pred) {
    int lo = 0, hi = n;
    while (hi > lo) {
        const int span = hi - lo;
        const int step = (span + 31) >> 5;
        const int p = lo + lane * step;
        const bool v = p < hi ? pred(p) : true;
        const uint32_t m = __ballot_sync(0xffffffffu, v);
        const int f = m ? __ffs(m) - 1 : 32;
        if (f == 0) return lo;
        const int new_hi = min(lo + f * step, hi);
        lo = lo + (f - 1) * step + 1;
        hi = new_hi;
    }
    return lo;
}

// CAND: additionally the cross-check's band candidates for |dy| <= inner (l2verify.cu): row arg-min candL[q] and, by 64-bit
// atomicMin, column arg-min candR[t] inside the inner band
template <int D, int MASK, bool CAND>
__global__ void __launch_bounds__(256, 4)
l2_band_kernel(Geom g, MatchParams mp, const uint32_t *__restrict__ counts, const float *__restrict__ fdesc,
               const float *__restrict__ kx, const float *__restrict__ ky, unsigned long long *__restrict__ best_out,
               unsigned long long *__restrict__ second_out, const int *__restrict__ rowstart, float inner,
               unsigned long long *__restrict__ candL, unsigned long long *__restrict__ candR) {
    const int pair = blockIdx.y;
    const int qi = 2 * pair, ti = 2 * pair + 1;
    const int nq = min((int)counts[qi], g.kp_cap), nt = min((int)counts[ti], g.kp_cap);
    const int lane = threadIdx.x & 31;
    const int qidx = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (qidx >= nq) return;
    const float *tkx = kx + (size_t)ti * g.kp_cap, *tky = ky + (size_t)ti * g.kp_cap;
    const float qx = kx[(size_t)qi * g.kp_cap + qidx];
    const float qy = __fadd_rn(ky[(size_t)qi * g.kp_cap + qidx], mp.q_off);
    // candidate rows from the train image's row table, trimmed to the exact allowed run
    const float reach = MASK == FE_MASK_EPIPOLAR ? mp.epi_threshold : mp.half_h;
    int lo, hi;
    band_range(rowstart + (size_t)ti * (g.rs_h + 2), g.rs_h, qy - mp.t_off, reach, lo, hi);
    hi = min(hi, nt);
    if (MASK == FE_MASK_EPIPOLAR)
        band_trim(lo, hi, lane, [&](int t) { return __fsub_rn(qy, __fadd_rn(tky[t], mp.t_off)) <= reach; },
                  [&](int t) { return __fsub_rn(qy, __fadd_rn(tky[t], mp.t_off)) < -reach; });
    else
        band_trim(lo, hi, lane, [&](int t) { return __fsub_rn(qy, __fadd_rn(tky[t], mp.t_off)) < reach; },
                  [&](int t) { return __fsub_rn(qy, __fadd_rn(tky[t], mp.t_off)) <= -reach; });
    // one candidate per iteration, the whole warp on its 512-byte row (coalesced); all lanes hold the result
    WarpRow<D> qr;
    qr.load(fdesc + ((size_t)qi * g.kp_cap + qidx) * 128, lane);
    unsigned long long best = KEY64_NONE, second = KEY64_NONE, inbest = KEY64_NONE;
    // the inner band is a contiguous sub-run of [lo, hi) (trains are raster-ordered): trim once, no coordinate reads in the loop
    int ilo = lo, ihi = hi;
    if (CAND)
        band_trim(ilo, ihi, lane, [&](int t) { return __fsub_rn(qy, __fadd_rn(tky[t], mp.t_off)) <= inner; },
                  [&](int t) { return __fsub_rn(qy, __fadd_rn(tky[t], mp.t_off)) < -inner; });
    if (MASK == FE_MASK_EPIPOLAR) {
        // 32 trains per round.  Every lane first forms ITS partial sum (its D / 32 dimensions) of all 32 trains -- the same
        // subtract / FMA chain as WarpRow::dist2 -- then a transposed reduction (xor 16, 8, 4, 2, 1: at every step a lane
        // keeps one half of its values and trades the other half) leaves lane l with the total of train l.  The additions form
        // exactly the butterfly's tree, so the bits equal WarpRow::dist2's; 31 shuffles per 32 distances instead of 160.
        const float *trow = fdesc + (size_t)ti * g.kp_cap * 128;
        // W = 32, 16 or 8 trains per round (a band holds ~36 trains: 32 + 8 instead of 2 x 32).  With W < 32 values per lane
        // the first steps (xor >= W) are plain butterfly additions of all W values, the halving starts at xor W / 2: the tree
        // is the same, lanes l and l ^ W (...) hold duplicates and only lanes < W act on the result.
        auto round = [&](auto wtag, int tb) {
            constexpr int W = decltype(wtag)::value;
            float part[W];
#pragma unroll
            for (int i = 0; i < W; ++i) {
                const float *row = trow + (size_t)min(tb + i, hi - 1) * 128;      // (the tail repeats the last train; ignored below)
                float tv[D / 32];
                if (D == 128) { const float4 v = __ldg(reinterpret_cast<const float4 *>(row) + lane); tv[0] = v.x; tv[1] = v.y; tv[D == 128 ? 2 : 0] = v.z; tv[D == 128 ? 3 : 1] = v.w; }
                else { const float2 v = __ldg(reinterpret_cast<const float2 *>(row) + lane); tv[0] = v.x; tv[1] = v.y; }
                float acc = 0.f;
#pragma unroll
                for (int d = 0; d < D / 32; ++d) { const float df = __fsub_rn(qr.q[d], tv[d]); acc = __fmaf_rn(df, df, acc); }
                part[i] = acc;
            }
#pragma unroll
            for (int off = 16; off; off >>= 1) {
                if (off >= W) {
#pragma unroll
                    for (int i = 0; i < W; ++i) part[i] = __fadd_rn(part[i], __shfl_xor_sync(0xffffffffu, part[i], off));
                } else {
                    const bool up = lane & off;
#pragma unroll
                    for (int i = 0; i < off; ++i) {
                        const float keep = up ? part[i + off] : part[i], send = up ? part[i] : part[i + off];
                        part[i] = __fadd_rn(keep, __shfl_xor_sync(0xffffffffu, send, off));
                    }
                }
            }
            const int t = tb + (lane & (W - 1));
            if (lane < W && t < hi) {
                const unsigned long long bits = (unsigned long long)__float_as_uint(part[0]) << 32;
                push2(best, second, bits | (unsigned)t);
                if (CAND && t >= ilo && t < ihi) {
                    inbest = min(inbest, bits | (unsigned)t);
                    atomicMin(&candR[(size_t)pair * g.kp_cap + t], bits | (unsigned)qidx);
                }
            }
        };
        int tb = lo;
        while (hi - tb > 16) { round(std::integral_constant<int, 32>{}, tb); tb += 32; }
        if (hi - tb > 8) { round(std::integral_constant<int, 16>{}, tb); tb += 16; }
        if (hi - tb > 0) round(std::integral_constant<int, 8>{}, tb);
        // merge the lanes' (best, second) pairs and inner-band minima: keys are distinct, so the result is the sequential one
#pragma unroll
        for (int off = 16; off; off >>= 1) {
            const unsigned long long ob = __shfl_xor_sync(0xffffffffu, best, off), os = __shfl_xor_sync(0xffffffffu, second, off);
            second = min(max(best, ob), min(second, os));
            best = min(best, ob);
            if (CAND) inbest = min(inbest, __shfl_xor_sync(0xffffffffu, inbest, off));
        }
    } else
    for (int t = lo; t < hi; ++t) {
        if (MASK == FE_MASK_WINDOW && !(fabsf(__fsub_rn(qx, tkx[t])) < mp.half_w)) continue;
        const float d2 = qr.dist2(fdesc + ((size_t)ti * g.kp_cap + t) * 128, lane);
        const unsigned long long bits = (unsigned long long)__float_as_uint(d2) << 32;
        push2(best, second, bits | (unsigned)t);
        if (CAND && t >= ilo && t < ihi) {
            inbest = min(inbest, bits | (unsigned)t);
            if (lane == 0) atomicMin(&candR[(size_t)pair * g.kp_cap + t], bits | (unsigned)qidx);
        }
    }
    if (lane == 0) {
        if (best_out) {
            best_out[(size_t)pair * g.kp_cap + qidx] = best;
            second_out[(size_t)pair * g.kp_cap + qidx] = second;
        }
        if (CAND) candL[(size_t)pair * g.kp_cap + qidx] = inbest;
    }
}

int launch_l2_band(const Geom &g, int n_pairs, int dim, const MatchParams &mp, const Buffers &b, const uint32_t *counts,
                   cudaStream_t s) {
    dim3 grid(div_up(g.kp_cap, 8), n_pairs);
#define FE_BAND_GO(D, MASK) l2_band_kernel<D, MASK, false><<<grid, 256, 0, s>>>(g, mp, counts, b.fdesc, b.kx, b.ky, b.best64, b.second64, b.rowstart, 0.f, nullptr, nullptr)
    launch_rowstart(g, b, counts, s);
    if (dim == 64) { if (mp.mask == FE_MASK_EPIPOLAR) FE_BAND_GO(64, FE_MASK_EPIPOLAR); else FE_BAND_GO(64, FE_MASK_WINDOW); }
    else { if (mp.mask == FE_MASK_EPIPOLAR) FE_BAND_GO(128, FE_MASK_EPIPOLAR); else FE_BAND_GO(128, FE_MASK_WINDOW); }
#undef FE_BAND_GO
    return 2;
}

// Epipolar band pass that also yields the cross-check's band candidates (b.vf_candL / b.vf_candR) for |dy| <= inner <=
// mp.epi_threshold.  write_knn: also the (best, second) of mode A (the band of mp); otherwise only the candidates.
int launch_l2_band_cand(const Geom &g, int n_pairs, int dim, const MatchParams &mp, float inner, bool write_knn, const Buffers &b,
                        const uint32_t *counts, cudaStream_t s) {
    dim3 grid(div_up(g.kp_cap, 8), n_pairs);
    cudaMemsetAsync(b.vf_candR, 0xFF, sizeof(unsigned long long) * (size_t)n_pairs * g.kp_cap, s);
    launch_rowstart(g, b, counts, s);
    unsigned long long *bo = write_knn ? b.best64 : nullptr, *so = write_knn ? b.second64 : nullptr;
    if (dim == 64) l2_band_kernel<64, FE_MASK_EPIPOLAR, true><<<grid, 256, 0, s>>>(g, mp, counts, b.fdesc, b.kx, b.ky, bo, so, b.rowstart, inner, b.vf_candL, b.vf_candR);
    else l2_band_kernel<128, FE_MASK_EPIPOLAR, true><<<grid, 256, 0, s>>>(g, mp, counts, b.fdesc, b.kx, b.ky, bo, so, b.rowstart, inner, b.vf_candL, b.vf_candR);
    return 2;
}

// ---- finalisation on 64-bit keys ---------------------------------------------------------------------
constexpr int LFIN = 1024;

__device__ __forceinline__ uint32_t block_excl_scan_1024b(uint32_t v, uint32_t *s_warp, uint32_t &total) {
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
        s_warp[lane] = wi - w;
        if (lane == 31) s_warp[32] = wi;
    }
    __syncthreads();
    const uint32_t r = s_warp[wid] + incl - v;
    total = s_warp[32];
    __syncthreads();
    return r;
}

__device__ __forceinline__ float key_dist(unsigned long long k) { return __fsqrt_rn(__uint_as_float((uint32_t)(k >> 32))); }

// Lowe ratio on the reported (sqrt) distances: d0 < ratio * d1 in double, like the reference.
__global__ void __launch_bounds__(LFIN)
l2_finalize_ratio_kernel(Geom g, double ratio, const uint32_t *__restrict__ counts,
                         const unsigned long long *__restrict__ best, const unsigned long long *__restrict__ second,
                         fe_match *__restrict__ out, uint32_t *__restrict__ n_out) {
    __shared__ uint32_t s_warp[33];
    const int pair = blockIdx.x;
    const int nq = min((int)counts[2 * pair], g.kp_cap);
    const unsigned long long *b = best + (size_t)pair * g.kp_cap, *s2 = second + (size_t)pair * g.kp_cap;
    fe_match *o = out + (size_t)pair * g.kp_cap;
    uint32_t offset = 0;
    for (int base = 0; base < nq; base += LFIN) {
        const int i = base + threadIdx.x;
        bool good = false;
        unsigned long long kb = KEY64_NONE;
        if (i < nq) {
            kb = b[i];
            const unsigned long long ks = s2[i];
            if (kb != KEY64_NONE) good = ks == KEY64_NONE || (double)key_dist(kb) < ratio * (double)key_dist(ks);
        }
        uint32_t total;
        const uint32_t pos = offset + block_excl_scan_1024b(good ? 1u : 0u, s_warp, total);
        if (good) {
            fe_match m;
            m.queryIdx = (uint32_t)i; m.trainIdx = (uint32_t)(kb & 0xFFFFFFFFu); m.imgIdx = 0; m.distance = key_dist(kb);
            o[pos] = m;
        }
        offset += total;
    }
    if (threadIdx.x == 0) n_out[pair] = offset;
}

__global__ void __launch_bounds__(LFIN)
l2_finalize_cross_kernel(Geom g, float max_dy, const uint32_t *__restrict__ counts,
                         const unsigned long long *__restrict__ allbest, const unsigned long long *__restrict__ colbest,
                         const float *__restrict__ ky, fe_match *__restrict__ out, uint32_t *__restrict__ n_out) {
    __shared__ uint32_t s_warp[33];
    const int pair = blockIdx.x;
    const int nq = min((int)counts[2 * pair], g.kp_cap), nt = min((int)counts[2 * pair + 1], g.kp_cap);
    const unsigned long long *ab = allbest + (size_t)pair * g.kp_cap, *cb = colbest + (size_t)pair * g.kp_cap;
    const float *qy = ky + (size_t)(2 * pair) * g.kp_cap, *ty = ky + (size_t)(2 * pair + 1) * g.kp_cap;
    fe_match *o = out + (size_t)pair * g.kp_cap;
    uint32_t offset = 0;
    for (int base = 0; base < nq; base += LFIN) {
        const int i = base + threadIdx.x;
        bool good = false;
        unsigned long long kb = KEY64_NONE;
        if (i < nq && nt > 0) {
            kb = ab[i];
            const uint32_t t = (uint32_t)(kb & 0xFFFFFFFFu);
            good = kb != KEY64_NONE && t < (uint32_t)nt && (uint32_t)(cb[t] & 0xFFFFFFFFu) == (uint32_t)i;   // (no key: a row the verification never touched)
            if (good && max_dy >= 0.f) good = fabsf(__fsub_rn(qy[i], ty[t])) <= max_dy;
        }
        uint32_t total;
        const uint32_t pos = offset + block_excl_scan_1024b(good ? 1u : 0u, s_warp, total);
        if (good) {
            fe_match m;
            m.queryIdx = (uint32_t)i; m.trainIdx = (uint32_t)(kb & 0xFFFFFFFFu); m.imgIdx = 0; m.distance = key_dist(kb);
            o[pos] = m;
        }
        offset += total;
    }
    if (threadIdx.x == 0) n_out[pair] = offset;
}

// liveGraph's tracker on float rows (/root/reference src/front_end/algorithm.py:1160-1190), the 64-bit-key twin of match.cu's
// finalize_cross_both_kernel: landmark i of the current frame continues landmark t of the previous one iff the row arg-mins
// of the left and of the right rows both name t and both column arg-mins name i.  Left distance; ordered by i.
__global__ void __launch_bounds__(LFIN)
l2_finalize_cross_both_kernel(Geom g, const uint32_t *__restrict__ counts, const unsigned long long *__restrict__ abL,
                              const unsigned long long *__restrict__ cbL, const unsigned long long *__restrict__ abR,
                              const unsigned long long *__restrict__ cbR, fe_match *__restrict__ out, uint32_t *__restrict__ n_out) {
    __shared__ uint32_t s_warp[33];
    const int pair = blockIdx.x;
    const int nq = min((int)counts[2 * pair], g.kp_cap), nt = min((int)counts[2 * pair + 1], g.kp_cap);
    const size_t o0 = (size_t)pair * g.kp_cap;
    fe_match *o = out + o0;
    uint32_t offset = 0;
    for (int base = 0; base < nq; base += LFIN) {
        const int i = base + threadIdx.x;
        bool good = false;
        unsigned long long kl = KEY64_NONE;
        if (i < nq && nt > 0) {
            kl = abL[o0 + i];
            const unsigned long long kr = abR[o0 + i];
            const uint32_t tl = (uint32_t)(kl & 0xFFFFFFFFu), tr = (uint32_t)(kr & 0xFFFFFFFFu);
            good = kl != KEY64_NONE && kr != KEY64_NONE && tl == tr && tl < (uint32_t)nt &&
                   (uint32_t)(cbL[o0 + tl] & 0xFFFFFFFFu) == (uint32_t)i && (uint32_t)(cbR[o0 + tr] & 0xFFFFFFFFu) == (uint32_t)i;
        }
        uint32_t total;
        const uint32_t pos = offset + block_excl_scan_1024b(good ? 1u : 0u, s_warp, total);
        if (good) {
            fe_match m;
            m.queryIdx = (uint32_t)i; m.trainIdx = (uint32_t)(kl & 0xFFFFFFFFu); m.imgIdx = 0; m.distance = key_dist(kl);
            o[pos] = m;
        }
        offset += total;
    }
    if (threadIdx.x == 0) n_out[pair] = offset;
}

template <int D>
static void launch_l2_d(const Geom &g, int n_pairs, const MatchParams &mp, bool masked, bool all, const Buffers &b,
                        const uint32_t *counts, cudaStream_t s) {
    const size_t smem = (size_t)2 * D * LPAD * sizeof(float);
    dim3 grid(div_up(g.kp_cap, LT), n_pairs);
#define FE_L2_GO(MASK, M, A)                                                                                   \
    do {                                                                                                       \
        cudaFuncSetAttribute(l2_match_kernel<D, MASK, M, A>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        l2_match_kernel<D, MASK, M, A><<<grid, 256, smem, s>>>(g, mp, counts, b.fdesc, b.kx, b.ky, b.best64, b.second64, \
                                                               b.allbest64, b.colbest64);                      \
    } while (0)
    if (masked) {
        if (mp.mask == FE_MASK_EPIPOLAR) FE_L2_GO(FE_MASK_EPIPOLAR, true, false);
        else if (mp.mask == FE_MASK_WINDOW) FE_L2_GO(FE_MASK_WINDOW, true, false);
        else FE_L2_GO(FE_MASK_NONE, true, false);
    }
    if (all) FE_L2_GO(FE_MASK_NONE, false, true);
#undef FE_L2_GO
}

int launch_l2_match(const Geom &g, int n_pairs, int dim, const MatchParams &mp, bool masked, bool all, const Buffers &b,
                    const uint32_t *counts, cudaStream_t s) {
    if (all) cudaMemsetAsync(b.colbest64, 0xFF, sizeof(unsigned long long) * (size_t)n_pairs * g.kp_cap, s);
    if (dim == 64) launch_l2_d<64>(g, n_pairs, mp, masked, all, b, counts, s);
    else launch_l2_d<128>(g, n_pairs, mp, masked, all, b, counts, s);
    return (masked ? 1 : 0) + (all ? 1 : 0);
}

int launch_l2_finalize_ratio(const Geom &g, int n_pairs, double ratio, const Buffers &b, const uint32_t *counts, cudaStream_t s) {
    l2_finalize_ratio_kernel<<<n_pairs, LFIN, 0, s>>>(g, ratio, counts, b.best64, b.second64, b.match_a, b.n_a);
    return 1;
}

int launch_l2_finalize_cross(const Geom &g, int n_pairs, float max_dy, const Buffers &b, const uint32_t *counts, cudaStream_t s) {
    l2_finalize_cross_kernel<<<n_pairs, LFIN, 0, s>>>(g, max_dy, counts, b.allbest64, b.colbest64, b.ky, b.match_b, b.n_b);
    return 1;
}

int launch_l2_finalize_cross_both(const Geom &g, int n_pairs, const uint32_t *counts, const unsigned long long *abL,
                                  const unsigned long long *cbL, const unsigned long long *abR, const unsigned long long *cbR,
                                  fe_match *out, uint32_t *n_out, cudaStream_t s) {
    l2_finalize_cross_both_kernel<<<n_pairs, LFIN, 0, s>>>(g, counts, abL, cbL, abR, cbR, out, n_out);
    return 1;
}

}  // namespace fe
