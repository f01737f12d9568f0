// SURF Fast-Hessian detector (cv::SURF::operator() with useProvidedKeypoints = false).
//
// Replaces /root/reference src/surf.cpp:167-206 (calcLayerDetAndTrace), :346-443 (findMaximaInLayer), :228-258
// (interpolateKeypoint) and the schedule of fastHessianDetector :462-512, reached from the services when the detector
// table selects "SURF" (src/front_end/features.py:149-156,441-453; src/utils.cpp:36-53).  The vendored CUDA twin
// src/cuda/surf.cu:204-526 has the same three steps; this is a fresh sm_100a formulation:
//   hessian_layer_kernel   one thread per sample of one scale-space layer: 10 box sums on the int32 integral image
//                          (3 Dxx + 3 Dyy + 4 Dxy boxes of the 9x9 pattern scaled to `size`), each (int sum) * float
//                          weight accumulated in double like calcHaarPattern, det = dx*dy - 0.81f*dxy*dxy (no FMA);
//                          the whole layer array is written (zeros outside the valid region), so no memset is needed;
//   hessian_maxima_kernel  one thread per interior sample of a middle layer: threshold, strict 26-neighbour NMS over
//                          (layer-1, layer, layer+1), 3-D quadratic interpolation with OpenCV 2.4's closed-form 3x3
//                          solve (Matx_FastSolveOp), atomic append of the accepted keypoint.
//   surf_rank_sort_kernel  std::sort(keypoints, KeypointGreater()) (src/surf.cpp:445-460,511) on the device: the comparator is
//                          a strict total order (response, size, octave, y, x), so the rank of a record -- the number of
//                          records that precede it -- is its final position; deterministic although the append order is not.
//   surf_raster_kernel     the batched pipeline's replacement of the sort: the maxima SURFInvoker keeps, in raster order
//                          (y, x, then KeypointGreater), bucketed by floor(y) -- what the banded matchers read.
// All of them take a batch of images; nothing returns to the host between detection and description.
#include "fe_internal.cuh"

namespace fe {

__global__ void __launch_bounds__(256)
hessian_layer_kernel(const int32_t *__restrict__ S0, size_t s_img_stride, int stride, int R, int C, HessianLayer hl,
                     float *__restrict__ det0, float *__restrict__ trace0, size_t l_img_stride) {
    const int j = blockIdx.x * 64 + (threadIdx.x & 63), i = blockIdx.y * 4 + (threadIdx.x >> 6);
    const int rows = R / hl.step, cols = C / hl.step;
    if (i >= rows || j >= cols) return;
    const int32_t *S = S0 + (size_t)blockIdx.z * s_img_stride;
    float *det = det0 + (size_t)blockIdx.z * l_img_stride, *trace = trace0 + (size_t)blockIdx.z * l_img_stride;
    float d = 0.f, t = 0.f;
    const int si = i - hl.margin, sj = j - hl.margin;
    if (hl.valid && si >= 0 && si < hl.samples_i && sj >= 0 && sj < hl.samples_j) {
        const int32_t *p = S + (size_t)(si * hl.step) * stride + sj * hl.step;
        auto haar = [&](int first, int n) {
            double acc = 0.0;
            for (int k = first; k < first + n; ++k) {
                const HaarBoxI &b = hl.box[k];
                const int v = p[b.dy1 * stride + b.dx1] + p[b.dy2 * stride + b.dx2] - p[b.dy2 * stride + b.dx1] - p[b.dy1 * stride + b.dx2];
                acc = __dadd_rn(acc, (double)__fmul_rn((float)v, b.w));
            }
            return (float)acc;
        };
        const float dx = haar(0, 3), dy = haar(3, 3), dxy = haar(6, 4);
        d = __fsub_rn(__fmul_rn(dx, dy), __fmul_rn(__fmul_rn(0.81f, dxy), dxy));
        t = __fadd_rn(dx, dy);
    }
    det[(size_t)i * cols + j] = d;
    trace[(size_t)i * cols + j] = t;
}

int launch_hessian_layer(const int32_t *S, size_t s_img_stride, int stride, int R, int C, const HessianLayer &hl, float *det,
                         float *trace, size_t l_img_stride, int n_images, cudaStream_t s) {
    dim3 grid(div_up(C / hl.step, 64), div_up(R / hl.step, 4), n_images);
    if (grid.x == 0 || grid.y == 0) return 0;
    hessian_layer_kernel<<<grid, 256, 0, s>>>(S, s_img_stride, stride, R, C, hl, det, trace, l_img_stride);
    return 1;
}

// Matx<float,3,3>::solve(b, DECOMP_LU) of OpenCV 2.4 (Matx_FastSolveOp<float,3,1>): Cramer's rule, plain float, no FMA
__device__ __forceinline__ float m2f(float p, float q, float r, float s) { return __fsub_rn(__fmul_rn(p, q), __fmul_rn(r, s)); }

__global__ void __launch_bounds__(256)
hessian_maxima_kernel(const float *__restrict__ d0, const float *__restrict__ d1, const float *__restrict__ d2,
                      const float *__restrict__ tr, size_t l_img_stride, int rows, int cols, int margin, int size, int size_prev,
                      int step, int octave, float threshold, fe_kpoint *__restrict__ out, int cap, uint32_t *__restrict__ count) {
    const int j = margin + blockIdx.x * 64 + (threadIdx.x & 63), i = margin + blockIdx.y * 4 + (threadIdx.x >> 6);
    if (i >= rows - margin || j >= cols - margin) return;
    const size_t lo = (size_t)blockIdx.z * l_img_stride;
    d0 += lo; d1 += lo; d2 += lo; tr += lo;
    out += (size_t)blockIdx.z * cap;
    count += blockIdx.z;
    const size_t o = (size_t)i * cols + j;
    const float val0 = d1[o];
    if (!(val0 > threshold)) return;
    float N9[3][9];
    const float *L[3] = {d0 + o, d1 + o, d2 + o};
#pragma unroll
    for (int l = 0; l < 3; ++l)
#pragma unroll
        for (int k = 0; k < 9; ++k) N9[l][k] = L[l][(k / 3 - 1) * cols + (k % 3 - 1)];
    bool is_max = true;
#pragma unroll
    for (int l = 0; l < 3; ++l)
#pragma unroll
        for (int k = 0; k < 9; ++k)
            if (!(l == 1 && k == 4)) is_max = is_max && (val0 > N9[l][k]);
    if (!is_max) return;
    const int sum_i = step * (i - (size / 2) / step), sum_j = step * (j - (size / 2) / step);
    float y = __fadd_rn((float)sum_i, __fmul_rn((float)(size - 1), 0.5f));
    float x = __fadd_rn((float)sum_j, __fmul_rn((float)(size - 1), 0.5f));
    float ksize = (float)size;
    // interpolateKeypoint
    const float b0 = -__fdiv_rn(__fsub_rn(N9[1][5], N9[1][3]), 2.f), b1 = -__fdiv_rn(__fsub_rn(N9[1][7], N9[1][1]), 2.f),
                b2 = -__fdiv_rn(__fsub_rn(N9[2][4], N9[0][4]), 2.f);
    const float axy = __fdiv_rn(__fadd_rn(__fsub_rn(__fsub_rn(N9[1][8], N9[1][6]), N9[1][2]), N9[1][0]), 4.f);
    const float axs = __fdiv_rn(__fadd_rn(__fsub_rn(__fsub_rn(N9[2][5], N9[2][3]), N9[0][5]), N9[0][3]), 4.f);
    const float ays = __fdiv_rn(__fadd_rn(__fsub_rn(__fsub_rn(N9[2][7], N9[2][1]), N9[0][7]), N9[0][1]), 4.f);
    const float axx = __fadd_rn(__fsub_rn(N9[1][3], __fmul_rn(2.f, N9[1][4])), N9[1][5]);
    const float ayy = __fadd_rn(__fsub_rn(N9[1][1], __fmul_rn(2.f, N9[1][4])), N9[1][7]);
    const float ass = __fadd_rn(__fsub_rn(N9[0][4], __fmul_rn(2.f, N9[1][4])), N9[2][4]);
    // rows of A: (axx axy axs), (axy ayy ays), (axs ays ass)
    float det = __fadd_rn(__fsub_rn(__fmul_rn(axx, m2f(ayy, ass, ays, ays)), __fmul_rn(axy, m2f(axy, ass, axs, ays))),
                          __fmul_rn(axs, m2f(axy, ays, axs, ayy)));
    float x0 = 0.f, x1 = 0.f, x2 = 0.f;
    if (det != 0.f) {
        det = __fdiv_rn(1.f, det);
        x0 = __fmul_rn(det, __fadd_rn(__fsub_rn(__fmul_rn(b0, m2f(ayy, ass, ays, ays)), __fmul_rn(axy, m2f(b1, ass, ays, b2))),
                                      __fmul_rn(axs, m2f(b1, ays, ayy, b2))));
        x1 = __fmul_rn(det, __fadd_rn(__fsub_rn(__fmul_rn(axx, m2f(b1, ass, ays, b2)), __fmul_rn(b0, m2f(axy, ass, ays, axs))),
                                      __fmul_rn(axs, m2f(axy, b2, b1, axs))));
        x2 = __fmul_rn(det, __fadd_rn(__fsub_rn(__fmul_rn(axx, m2f(ayy, b2, b1, ays)), __fmul_rn(axy, m2f(axy, b2, b1, axs))),
                                      __fmul_rn(b0, m2f(axy, ays, ayy, axs))));
    }
    const bool ok = (x0 != 0.f || x1 != 0.f || x2 != 0.f) && fabsf(x0) <= 1.f && fabsf(x1) <= 1.f && fabsf(x2) <= 1.f;
    if (!ok) return;
    x = __fadd_rn(x, __fmul_rn(x0, (float)step));
    y = __fadd_rn(y, __fmul_rn(x1, (float)step));
    ksize = (float)__float2int_rn(__fadd_rn(ksize, __fmul_rn(x2, (float)(size - size_prev))));
    const uint32_t pos = atomicAdd(count, 1u);
    if (pos < (uint32_t)cap) {
        const float t = tr[o];
        fe_kpoint k;
        k.x = x; k.y = y; k.size = ksize; k.angle = -1.f; k.response = val0; k.octave = octave;
        k.class_id = t > 0.f ? 1 : (t < 0.f ? -1 : 0);        // CV_SIGN(trace): sign of the Laplacian
        out[pos] = k;
    }
}

int launch_hessian_maxima(const float *d0, const float *d1, const float *d2, const float *tr, size_t l_img_stride, int rows,
                          int cols, int margin, int size, int size_prev, int step, int octave, float threshold, fe_kpoint *out,
                          int cap, uint32_t *count, int n_images, cudaStream_t s) {
    if (rows - 2 * margin <= 0 || cols - 2 * margin <= 0) return 0;
    dim3 grid(div_up(cols - 2 * margin, 64), div_up(rows - 2 * margin, 4), n_images);
    hessian_maxima_kernel<<<grid, 256, 0, s>>>(d0, d1, d2, tr, l_img_stride, rows, cols, margin, size, size_prev, step, octave,
                                               threshold, out, cap, count);
    return 1;
}

// KeypointGreater (src/surf.cpp:445-460): response, size, octave descending, then y descending, x ASCENDING-is-greater
__device__ __forceinline__ bool kp_greater(const fe_kpoint &a, const fe_kpoint &q) {
    if (a.response > q.response) return true;
    if (a.response < q.response) return false;
    if (a.size > q.size) return true;
    if (a.size < q.size) return false;
    if (a.octave > q.octave) return true;
    if (a.octave < q.octave) return false;
    if (a.y < q.y) return false;
    if (a.y > q.y) return true;
    return a.x < q.x;
}

__global__ void __launch_bounds__(256)
surf_rank_sort_kernel(const fe_kpoint *__restrict__ in, fe_kpoint *__restrict__ out, const uint32_t *__restrict__ count, int cap,
                      uint32_t *__restrict__ max_size_bits) {
    __shared__ fe_kpoint s_tile[256];
    const int image = blockIdx.y;
    const int n = min((int)count[image], cap);
    if (blockIdx.x * 256 >= n) return;
    const fe_kpoint *src = in + (size_t)image * cap;
    const int i = blockIdx.x * 256 + threadIdx.x;
    fe_kpoint me{};
    if (i < n) me = src[i];
    int rank = 0;
    for (int t0 = 0; t0 < n; t0 += 256) {
        __syncthreads();
        if (t0 + (int)threadIdx.x < n) s_tile[threadIdx.x] = src[t0 + threadIdx.x];
        __syncthreads();
        const int tn = min(256, n - t0);
        if (i < n)
            for (int k = 0; k < tn; ++k) rank += kp_greater(s_tile[k], me) ? 1 : 0;
    }
    if (i < n) {
        out[(size_t)image * cap + rank] = me;
        atomicMax(&max_size_bits[image], __float_as_uint(fmaxf(me.size, 0.f)));
    }
}

int launch_surf_rank_sort(const fe_kpoint *in, fe_kpoint *out, const uint32_t *count, int cap, uint32_t *max_size_bits, int n_images,
                          cudaStream_t s) {
    cudaMemsetAsync(max_size_bits, 0, sizeof(uint32_t) * n_images, s);
    dim3 grid(div_up(cap, 256), n_images);
    surf_rank_sort_kernel<<<grid, 256, 0, s>>>(in, out, count, cap, max_size_bits);
    return 1;
}

// ---- batched pipeline: the maxima that survive SURFInvoker, in raster order ---------------------------------------------
// The banded matchers need keypoints whose floor(y) never decreases; the maxima arrive in atomic-append order.  One CTA per
// image, everything in shared memory: survivor bits and a histogram of floor(y) (pass 1), an exclusive scan of the histogram,
// a scatter of survivor indices into their rows (pass 2), and a rank inside each row (pass 3, ~16 keypoints per row at
// 1280x720) under the strict total order (y, x, KeypointGreater) -- deterministic although the append order is not.
constexpr int RASTER_THREADS = 1024;

__device__ __forceinline__ int raster_row(float y, int h) { return min(max((int)floorf(y), 0), h - 1); }

// a precedes q in the batch's order; the input index breaks ties of identical records (whose bytes are then the same anyway)
__device__ __forceinline__ bool raster_before(const fe_kpoint &a, int ia, const fe_kpoint &q, int iq) {
    if (a.y != q.y) return a.y < q.y;
    if (a.x != q.x) return a.x < q.x;
    if (kp_greater(a, q)) return true;
    if (kp_greater(q, a)) return false;
    return ia < iq;
}

size_t surf_raster_smem(int kp_cap, int h) {
    return sizeof(uint32_t) * div_up(kp_cap, 32) + sizeof(int) * (size_t)(h + 1) + sizeof(uint16_t) * (size_t)kp_cap;
}

__global__ void __launch_bounds__(RASTER_THREADS)
surf_raster_kernel(const fe_kpoint *__restrict__ in, const uint32_t *__restrict__ count, Geom g, int upright,
                   fe_kpoint *__restrict__ out, float *__restrict__ kx, float *__restrict__ ky, uint32_t *__restrict__ n_out) {
    extern __shared__ __align__(16) uint32_t s_raster[];
    const int image = blockIdx.x, cap = g.kp_cap, H = g.h, tid = threadIdx.x;
    const int words = div_up(cap, 32);
    uint32_t *keep = s_raster;                                        // [words] survivor bits
    int *rows = reinterpret_cast<int *>(keep + words);                // [H + 1] counts -> starts -> ends of the rows
    uint16_t *order = reinterpret_cast<uint16_t *>(rows + H + 1);     // [cap] input index of the survivors, row by row
    const uint32_t found = count[image];
    const int n = min((int)found, cap);
    const fe_kpoint *src = in + (size_t)image * cap;
    for (int i = tid; i < words; i += RASTER_THREADS) keep[i] = 0u;
    for (int r = tid; r <= H; r += RASTER_THREADS) rows[r] = 0;
    __syncthreads();
    for (int i = tid; i < n; i += RASTER_THREADS) {
        const fe_kpoint k = src[i];
        if (!surf_drops(k.x, k.y, k.size, g.w, g.h, upright != 0, SURF_DIRECT_MAX_WIN)) {
            atomicOr(&keep[i >> 5], 1u << (i & 31));
            atomicAdd(&rows[raster_row(k.y, H)], 1);
        }
    }
    __syncthreads();
    {   // exclusive scan of rows[0 .. H]: every thread owns a contiguous run of `per` rows
        __shared__ int s_warp[RASTER_THREADS / 32];
        const int per = div_up(H + 1, RASTER_THREADS), r0 = min(tid * per, H + 1), r1 = min(r0 + per, H + 1);
        int local = 0;
        for (int r = r0; r < r1; ++r) local += rows[r];
        const int lane = tid & 31, warp = tid >> 5;
        int incl = local;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            int w = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += v;
            }
            s_warp[lane] = w;
        }
        __syncthreads();
        int run = (warp > 0 ? s_warp[warp - 1] : 0) + incl - local;
        for (int r = r0; r < r1; ++r) { const int c = rows[r]; rows[r] = run; run += c; }
    }
    __syncthreads();
    const int m = rows[H];                   // survivors (row H is empty: its start is the total)
    for (int i = tid; i < n; i += RASTER_THREADS)
        if (keep[i >> 5] & (1u << (i & 31))) order[atomicAdd(&rows[raster_row(src[i].y, H)], 1)] = (uint16_t)i;
    __syncthreads();                         // rows[r] is now the end of row r, the start of row r + 1
    fe_kpoint *dst = out + (size_t)image * cap;
    float *dx = kx + (size_t)image * cap, *dy = ky + (size_t)image * cap;
    for (int p = tid; p < m; p += RASTER_THREADS) {
        const int i = order[p];
        const fe_kpoint k = src[i];
        const int r = raster_row(k.y, H), lo = r > 0 ? rows[r - 1] : 0, hi = rows[r];
        int rank = 0;
        for (int q = lo; q < hi; ++q) {
            const int j = order[q];
            if (j != i && raster_before(src[j], j, k, i)) ++rank;
        }
        dst[lo + rank] = k;
        dx[lo + rank] = k.x;
        dy[lo + rank] = k.y;
    }
    if (found > (uint32_t)cap) {
        // more maxima than capacity (the caller reports FE_ERR_CAPACITY): the consumers read all cap records, so the tail
        // holds empty records below the last row -- still raster-ordered, dropped by the descriptor pass
        fe_kpoint e{};
        e.y = (float)H; e.angle = -1.f;
        for (int p = m + tid; p < cap; p += RASTER_THREADS) { dst[p] = e; dx[p] = 0.f; dy[p] = e.y; }
    }
    if (tid == 0) n_out[image] = found > (uint32_t)cap ? found : (uint32_t)m;
}

int launch_surf_raster(const Geom &g, const fe_kpoint *in, const uint32_t *count, bool upright, const Buffers &b, cudaStream_t s) {
    const size_t smem = surf_raster_smem(g.kp_cap, g.h);
    if (smem > 48 * 1024) cudaFuncSetAttribute(surf_raster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    surf_raster_kernel<<<g.n_images, RASTER_THREADS, smem, s>>>(in, count, g, upright ? 1 : 0, b.kp, b.kx, b.ky, b.n_kp);
    return 1;
}

}  // namespace fe
