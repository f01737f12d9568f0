// WindowMatcher over a device-resident sequence of stereo frames.
//
// Replaces WindowMatcher::newStereo's data-parallel part (/root/reference src/WindowMatcher.cpp:75-231):
//   * every stereo match of a frame becomes a landmark (:79-85), triangulated with Q * [xl, yl, xl - xr, 1]
//     and divided by 1000 * w (:36-51);
//   * consecutive frames only: landmarks(cur) vs landmarks(prev), search-box mask on the LEFT keypoint
//     coordinates (:104-128), left descriptors (:134-148), kNN-2 (:150-153), Lowe 0.8 with singleton
//     acceptance (:161-224); queryIdx / trainIdx index the landmark lists (:227-231).
// The landmark lists are gathered on the device from the batched pipeline's own outputs (matches_a rows of
// pair f = landmarks of frame f), laid out as "virtual pairs" v = (cur = frame v + 1, prev = frame v) so that
// the stereo matcher's kernels (banded kNN-2 + ratio finalisation) run unchanged on them.  Landmarks keep the
// order of matches_a (ascending left keypoint index = raster order), so the banded kernel's precondition holds.
// SURF batches gather float rows instead (the first 64 / 128 floats of every fdesc row), which the L2 matchers read.
#include "fe_internal.cuh"

namespace fe {

// Row copies of the landmark kernels: LANES threads per row, `part` = the thread's share of it.
// 32-byte binary rows (ORB-256), one thread each.
struct BinRows {
    static constexpr int LANES = 1;
    const uint8_t *src;
    uint8_t *dst;
    __device__ __forceinline__ void copy(size_t d, size_t s, int) const {
        const uint4 *sd = reinterpret_cast<const uint4 *>(src + s * 32);
        uint4 *dd = reinterpret_cast<uint4 *>(dst + d * 32);
        dd[0] = __ldg(sd); dd[1] = __ldg(sd + 1);
    }
};
// The first D floats of a 128-float fdesc row (SURF-64 / SURF-128) to a row DST floats apart, one float4 per thread.
template <int D, int DST>
struct FloatRows {
    static constexpr int LANES = D / 4;
    const float *src;
    float *dst;
    __device__ __forceinline__ void copy(size_t d, size_t s, int part) const {
        reinterpret_cast<float4 *>(dst + d * DST)[part] = __ldg(reinterpret_cast<const float4 *>(src + s * 128) + part);
    }
};

template <typename Rows>
__global__ void __launch_bounds__(256)
gather_landmarks_kernel(Geom g, int side, const uint32_t *__restrict__ n_a, const fe_match *__restrict__ match_a, Rows rows,
                        const float *__restrict__ kx, const float *__restrict__ ky, float *__restrict__ wkx,
                        float *__restrict__ wky, uint32_t *__restrict__ wcount) {
    const int v = blockIdx.y, s = blockIdx.z;           // virtual pair, slot (0 = current / query, 1 = previous / train)
    const int frame = v + 1 - s;
    const int n = min((int)n_a[frame], g.kp_cap);
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = t / Rows::LANES, part = t % Rows::LANES;
    const size_t slot = (size_t)(2 * v + s);
    if (t == 0) wcount[slot] = (uint32_t)n;
    if (i >= n) return;
    const fe_match mt = match_a[(size_t)frame * g.kp_cap + i];
    const uint32_t q = side ? mt.trainIdx : mt.queryIdx;                     // left (right) keypoint of landmark i
    const size_t src = (size_t)(2 * frame + side) * g.kp_cap + q, dst = slot * g.kp_cap + i;
    rows.copy(dst, src, part);
    if (wkx && part == 0) { wkx[dst] = kx[src]; wky[dst] = ky[src]; }
}

template <typename Rows>
static int gather_go(const Geom &g, int n_frames, const Buffers &b, int side, Rows rows, float *wkx, float *wky,
                     uint32_t *wcount, cudaStream_t s) {
    dim3 grid(div_up(g.kp_cap * Rows::LANES, 256), n_frames - 1, 2);
    gather_landmarks_kernel<Rows><<<grid, 256, 0, s>>>(g, side, b.n_a, b.match_a, rows, b.kx, b.ky, wkx, wky, wcount);
    return 1;
}

int launch_gather_landmarks(const Geom &g, int n_frames, const Buffers &b, int side, uint8_t *wdesc, float *wkx, float *wky,
                            uint32_t *wcount, cudaStream_t s) {
    return gather_go(g, n_frames, b, side, BinRows{b.desc, wdesc}, wkx, wky, wcount, s);
}

int launch_gather_landmarks(const Geom &g, int n_frames, const Buffers &b, int side, int dim, float *wfdesc, float *wkx,
                            float *wky, uint32_t *wcount, cudaStream_t s) {
    if (dim == 64) return gather_go(g, n_frames, b, side, FloatRows<64, 128>{b.fdesc, wfdesc}, wkx, wky, wcount, s);
    return gather_go(g, n_frames, b, side, FloatRows<128, 128>{b.fdesc, wfdesc}, wkx, wky, wcount, s);
}

// Q * [xl, yl, xl - xr, 1] / (1000 * w), double precision, products summed left to right without FMA.
__global__ void __launch_bounds__(256)
triangulate_kernel(Geom g, const uint32_t *__restrict__ n_a, const fe_match *__restrict__ match_a,
                   const float *__restrict__ kx, const float *__restrict__ ky, const double *__restrict__ Q,
                   double *__restrict__ xyz) {
    const int frame = blockIdx.y;
    const int n = min((int)n_a[frame], g.kp_cap);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const fe_match m = match_a[(size_t)frame * g.kp_cap + i];
    const size_t l = (size_t)(2 * frame) * g.kp_cap + m.queryIdx, r = (size_t)(2 * frame + 1) * g.kp_cap + m.trainIdx;
    const double in[4] = {(double)kx[l], (double)ky[l], (double)__fsub_rn(kx[l], kx[r]), 1.0};
    double h[4];
#pragma unroll
    for (int row = 0; row < 4; ++row) {
        double acc = __dmul_rn(Q[row * 4], in[0]);
#pragma unroll
        for (int k = 1; k < 4; ++k) acc = __dadd_rn(acc, __dmul_rn(Q[row * 4 + k], in[k]));
        h[row] = acc;
    }
    const double den = __dmul_rn(1000.0, h[3]);
    double *o = xyz + ((size_t)frame * g.kp_cap + i) * 3;
    o[0] = __ddiv_rn(h[0], den); o[1] = __ddiv_rn(h[1], den); o[2] = __ddiv_rn(h[2], den);
}

int launch_triangulate(const Geom &g, int n_frames, const Buffers &b, const double *Q, double *xyz, cudaStream_t s) {
    dim3 grid(div_up(g.kp_cap, 256), n_frames);
    triangulate_kernel<<<grid, 256, 0, s>>>(g, b.n_a, b.match_a, b.kx, b.ky, Q, xyz);
    return 1;
}

// stereoLandmarks packing (/root/reference src/front_end/algorithm.py:893-913): for match i of a pair, the left
// keypoint / descriptor at queryIdx and the right ones at trainIdx are compacted to row i, and the match itself is
// re-indexed to (i, i, 0, distance).  Rows::LANES threads per match: 32-byte rBRIEF rows, or SURF float rows.
template <typename Rows>
__global__ void __launch_bounds__(256)
pack_landmarks_kernel(Geom g, const uint32_t *__restrict__ n_m, const fe_match *__restrict__ matches,
                      const fe_kpoint *__restrict__ kp, Rows lrows, Rows rrows, fe_kpoint *__restrict__ lkp,
                      fe_kpoint *__restrict__ rkp, fe_match *__restrict__ out) {
    const int pair = blockIdx.y;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = t / Rows::LANES, part = t % Rows::LANES;
    if (i >= min((int)n_m[pair], g.kp_cap)) return;
    const size_t o = (size_t)pair * g.kp_cap + i;
    const fe_match m = matches[o];
    const size_t l = (size_t)(2 * pair) * g.kp_cap + m.queryIdx, r = (size_t)(2 * pair + 1) * g.kp_cap + m.trainIdx;
    lrows.copy(o, l, part);
    rrows.copy(o, r, part);
    if (part) return;
    lkp[o] = kp[l];
    rkp[o] = kp[r];
    fe_match mo;
    mo.queryIdx = (uint32_t)i; mo.trainIdx = (uint32_t)i; mo.imgIdx = 0; mo.distance = m.distance;
    out[o] = mo;
}

template <typename Rows>
static int pack_go(const Geom &g, int n_pairs, const Buffers &b, const uint32_t *n_m, const fe_match *matches, fe_kpoint *lkp,
                   fe_kpoint *rkp, Rows lrows, Rows rrows, fe_match *out, cudaStream_t s) {
    dim3 grid(div_up(g.kp_cap * Rows::LANES, 256), n_pairs);
    pack_landmarks_kernel<Rows><<<grid, 256, 0, s>>>(g, n_m, matches, b.kp, lrows, rrows, lkp, rkp, out);
    return 1;
}

int launch_pack_landmarks(const Geom &g, int n_pairs, const Buffers &b, const uint32_t *n_m, const fe_match *matches,
                          fe_kpoint *lkp, fe_kpoint *rkp, uint8_t *ldesc, uint8_t *rdesc, fe_match *out, cudaStream_t s) {
    return pack_go(g, n_pairs, b, n_m, matches, lkp, rkp, BinRows{b.desc, ldesc}, BinRows{b.desc, rdesc}, out, s);
}

int launch_pack_landmarks(const Geom &g, int n_pairs, const Buffers &b, const uint32_t *n_m, const fe_match *matches,
                          fe_kpoint *lkp, fe_kpoint *rkp, int dim, float *ldesc, float *rdesc, fe_match *out, cudaStream_t s) {
    if (dim == 64)
        return pack_go(g, n_pairs, b, n_m, matches, lkp, rkp, FloatRows<64, 64>{b.fdesc, ldesc}, FloatRows<64, 64>{b.fdesc, rdesc}, out, s);
    return pack_go(g, n_pairs, b, n_m, matches, lkp, rkp, FloatRows<128, 128>{b.fdesc, ldesc}, FloatRows<128, 128>{b.fdesc, rdesc},
                   out, s);
}

}  // namespace fe
