// ORB orientation (intensity centroid), the descriptor's 7x7 float Gaussian, and rBRIEF-256.
//
// Replaces the tail of cv::ORB::detect (IC_Angle) and DescriptorExtractor::compute with ORB, as the
// reference reaches them at /root/reference bin/feature_node:50-54, src/front_end/features.py:450-451,
// 721-722, bin/detect_node:50-51, src/StereoCamera.cpp:84-89,123-128.  Semantics SURVEY.md A.3/A.4:
//   * m10 = sum u*I, m01 = sum v*I over |u| <= umax[|v|], radius 15; angle = fastAtan2(m01, m10) with
//     OpenCV's f32 degree-7 polynomial, evaluated WITHOUT fused multiply-add (pinned against cv2);
//   * blur = separable 7-tap sigma=2 in f32, BORDER_REFLECT_101, row pass as a left-to-right FMA
//     chain, column pass centre-out with pair sums, round-half-even to u8;
//   * bit i of the descriptor = blurred(p_2i rotated) < blurred(p_2i+1 rotated), rotation by
//     (cos, sin) of the angle in f32 (cos/sin taken in double, rounded to f32), coordinates rounded
//     half-even.
// The library is compiled with -fmad=false; every FMA below is explicit.
#include "fe_internal.cuh"

namespace fe {

// ORB's bit_pattern_31_ (256 tests x (x0, y0, x1, y1)).  Global, not __constant__: the CTA copies it
// to shared memory with per-thread distinct addresses, which the constant cache would serialise.
__device__ int8_t d_pattern[256][4] = {
#include "orb_pattern.inc"
};

__device__ __forceinline__ int reflect101(int i, int n) {
    if (i < 0) i = -i;
    if (i >= n) i = 2 * (n - 1) - i;
    return i;
}

constexpr int ORB_PATCH = 31;               // ORB's default patchSize: bit_pattern_31_ and the radius-15 intensity-centroid disc
constexpr int ORI_R = ORB_PATCH / 2;
constexpr int ORI_WARPS = 8;
constexpr int ORI_KPW = 8;                  // keypoints per warp (amortises the weight-table copy)
constexpr int ORI_WORDS = 9;                // 31 columns + up to 3 alignment bytes -> 9 words per patch row
constexpr int ORI_SLOTS = ORB_PATCH * ORI_WORDS;   // 279 (row, word) slots per keypoint, 9 rounds of 32 lanes
constexpr int ORI_K = (ORI_SLOTS + 31) / 32;       // slots per lane

__device__ __forceinline__ int dp4a_u8s8(uint32_t a, uint32_t b, int c) {
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// The radius-15 disc is read as aligned 32-bit words (31 rows x 9 words) instead of 709 byte gathers, and the moments are
// integer dot products: for word slot (row v, word w) and alignment off = (x - 15) & 3, byte b is column u = 4w + b - off - 15;
// the tables hold u (as s8, 0 outside the disc |u| <= umax[|v|]) and the 0/1 membership mask, so  m10 += dp4a(word, U)  and
// m01 += v * dp4a(word, M).  Integer arithmetic: the moments are bit-identical to the byte loop.  Built at compile time.
struct __align__(16) OriTables { uint32_t u[4][288], m[4][288]; };
constexpr OriTables make_ori_tables() {
    constexpr int umax[ORI_R + 1] = {15, 15, 15, 15, 14, 14, 14, 13, 13, 12, 11, 10, 9, 8, 6, 3};   // OpenCV's umax, radius 15
    OriTables t{};
    for (int off = 0; off < 4; ++off)
        for (int slot = 0; slot < ORI_SLOTS; ++slot) {
            const int r = slot / ORI_WORDS, w = slot - r * ORI_WORDS;
            const int v = r - ORI_R, d = umax[v < 0 ? -v : v];
            for (int b = 0; b < 4; ++b) {
                const int u = 4 * w + b - off - ORI_R;
                if (u >= -d && u <= d) { t.u[off][slot] |= (uint32_t)(u & 0xFF) << (8 * b); t.m[off][slot] |= 1u << (8 * b); }
            }
        }
    return t;
}
__device__ const OriTables d_ori_tab = make_ori_tables();

// Per-lane slot geometry, the same for every keypoint: slot lane + 32 k is (row r, word w) of the patch, at offset
// r * row_stride + w * word_stride from its first word, and row v = r - 15 of the disc
__device__ __forceinline__ void ori_slots(int lane, int row_stride, int word_stride, int (&soff)[ORI_K], int (&sv)[ORI_K]) {
#pragma unroll
    for (int k = 0; k < ORI_K; ++k) {
        const int slot = min(lane + 32 * k, ORI_SLOTS - 1);
        const int r = slot / ORI_WORDS, w = slot - r * ORI_WORDS;
        soff[k] = r * row_stride + w * word_stride;
        sv[k] = r - ORI_R;
    }
}

// Intensity-centroid angles (degrees, cv::fastAtan2) of two keypoints, one warp: words(k) gives this lane's words of slot
// lane + 32 k of both patches (0 past the last slot), whose alignments are off0 and off1; tu / tm are the weight tables
template <class Words>
__device__ __forceinline__ float2 ori_angles(Words words, int off0, int off1, const uint32_t (*tu)[288], const uint32_t (*tm)[288],
                                             const int (&sv)[ORI_K], int lane) {
    int m10a = 0, m01a = 0, m10b = 0, m01b = 0;
#pragma unroll
    for (int k = 0; k < ORI_K; ++k) {
        const int slot = min(lane + 32 * k, ORI_SLOTS - 1);
        const uint2 w = words(k);
        m10a = dp4a_u8s8(w.x, tu[off0][slot], m10a);
        m01a += sv[k] * dp4a_u8s8(w.x, tm[off0][slot], 0);
        m10b = dp4a_u8s8(w.y, tu[off1][slot], m10b);
        m01b += sv[k] * dp4a_u8s8(w.y, tm[off1][slot], 0);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        m10a += __shfl_xor_sync(0xffffffffu, m10a, o);
        m01a += __shfl_xor_sync(0xffffffffu, m01a, o);
        m10b += __shfl_xor_sync(0xffffffffu, m10b, o);
        m01b += __shfl_xor_sync(0xffffffffu, m01b, o);
    }
    return make_float2(fast_atan2_deg((float)m01a, (float)m10a), fast_atan2_deg((float)m01b, (float)m10b));
}

// The detector's keypoint record at index o (cv::KeyPoint of cv::ORB::detect: octave 0, class_id -1, the FAST score as
// response when reported), its float coordinates and its steering (cos, sin)
__device__ __forceinline__ void store_keypoint(size_t o, uint32_t key, float angle, float2 cs, float kp_size,
                                               const uint8_t *__restrict__ kp_score, int report_score, fe_kpoint *__restrict__ kp,
                                               float *__restrict__ kx, float *__restrict__ ky, float2 *__restrict__ kcs) {
    const int x = key & 0xFFFF, y = key >> 16;
    fe_kpoint k;
    k.x = (float)x; k.y = (float)y; k.size = kp_size; k.angle = angle;
    k.response = report_score ? (float)kp_score[o] : 0.f;
    k.octave = 0; k.class_id = -1;
    kp[o] = k;
    kx[o] = (float)x; ky[o] = (float)y;
    kcs[o] = cs;
}

// One warp per keypoint, the disc's words loaded straight from the image (rows coalesced).  Writes the wire-format keypoint,
// float coordinates and the steering (cos, sin).
__global__ void __launch_bounds__(ORI_WARPS * 32)
orient_pack_kernel(const uint8_t *__restrict__ img, Geom g, const uint32_t *__restrict__ n_kp,
                   const uint32_t *__restrict__ kp_key, const uint8_t *__restrict__ kp_score,
                   int orientation, int report_score, float kp_size, fe_kpoint *__restrict__ kp,
                   float *__restrict__ kx, float *__restrict__ ky, float2 *__restrict__ kcs) {
    __shared__ OriTables s_tab;
    const int image = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = min((int)n_kp[image], g.kp_cap);
    if (blockIdx.x * (ORI_WARPS * ORI_KPW) >= n) return;
    if (orientation) {          // the moments read the weight tables once per slot: from shared memory
        for (int i = threadIdx.x; i < (int)(sizeof(OriTables) / 16); i += ORI_WARPS * 32)
            reinterpret_cast<uint4 *>(&s_tab)[i] = reinterpret_cast<const uint4 *>(&d_ori_tab)[i];
        __syncthreads();
    }
    // per-lane slot geometry is the same for every keypoint: hoist it out of the keypoint loop
    int soff[ORI_K], sv[ORI_K];
    ori_slots(lane, g.pitch, 4, soff, sv);
    // lane `it` keeps keypoint `it` of this warp: the record, the double-precision cos / sin (the long pole of
    // the old kernel when evaluated by one lane per keypoint) and the stores are then done by 8 lanes at once
    uint32_t my_key = 0;
    float my_angle = -1.f;
    int my_n = 0;
    {   // one load brings the warp's keys: the keypoint loop then starts every round with its addresses known
        const int i = (blockIdx.x * ORI_KPW + lane) * ORI_WARPS + warp;
        if (lane < ORI_KPW && i < n) my_key = kp_key[(size_t)image * g.kp_cap + i];
    }
    // two keypoints per round: the 2 x 9 word loads are issued before any of them is consumed (the kernel is bound by the
    // latency of those loads, not by instruction issue)
    static_assert(ORI_KPW % 2 == 0, "keypoints are taken in pairs");
#pragma unroll 1
    for (int it = 0; it < ORI_KPW; it += 2) {
        const int i0 = (blockIdx.x * ORI_KPW + it) * ORI_WARPS + warp;
        if (i0 >= n) break;
        const bool two = i0 + ORI_WARPS < n;
        const uint32_t key0 = __shfl_sync(0xffffffffu, my_key, it);
        const uint32_t key1 = two ? __shfl_sync(0xffffffffu, my_key, it + 1) : key0;
        float2 angles = make_float2(-1.f, -1.f);
        if (orientation) {
            const int xl0 = (int)(key0 & 0xFFFF) - ORI_R, xa0 = xl0 & ~3;
            const int xl1 = (int)(key1 & 0xFFFF) - ORI_R, xa1 = xl1 & ~3;
            const uint8_t *base0 = img + (size_t)image * g.img_stride + (size_t)((int)(key0 >> 16) - ORI_R) * g.pitch + xa0;
            const uint8_t *base1 = img + (size_t)image * g.img_stride + (size_t)((int)(key1 >> 16) - ORI_R) * g.pitch + xa1;
            uint32_t wa[ORI_K], wb[ORI_K];
#pragma unroll
            for (int k = 0; k < ORI_K; ++k) {
                const bool in = lane + 32 * k < ORI_SLOTS;
                wa[k] = in ? __ldg(reinterpret_cast<const uint32_t *>(base0 + soff[k])) : 0u;
                wb[k] = in ? __ldg(reinterpret_cast<const uint32_t *>(base1 + soff[k])) : 0u;
            }
            angles = ori_angles([&](int k) { return make_uint2(wa[k], wb[k]); }, xl0 - xa0, xl1 - xa1, s_tab.u, s_tab.m, sv, lane);
        }
        if (lane == it) my_angle = angles.x;
        if (two && lane == it + 1) my_angle = angles.y;
        my_n = two ? it + 2 : it + 1;
    }
    if (lane < my_n) {
        const int i = (blockIdx.x * ORI_KPW + lane) * ORI_WARPS + warp;
        store_keypoint((size_t)image * g.kp_cap + i, my_key, my_angle, orientation ? steer(my_angle) : make_float2(1.f, 0.f),
                       kp_size, kp_score, report_score, kp, kx, ky, kcs);
    }
}

// General intensity-centroid orientation: any patch size (radius = patchSize / 2, OpenCV's umax table) and keypoints
// closer to the border than the radius (edgeThreshold < 16): cv::ORB computes IC_Angle on its bordered pyramid buffer,
// i.e. pixels outside the image are the raw BORDER_REFLECT_101 pixels (pinned against cv2 for edge 5 / 15 / 25 and
// patch 10 / 30 / 50).  One warp per keypoint, byte gathers; the fast path above serves the default 31-px patch.
__global__ void __launch_bounds__(ORI_WARPS * 32)
orient_general_kernel(const uint8_t *__restrict__ img, Geom g, const uint32_t *__restrict__ n_kp,
                      const uint32_t *__restrict__ kp_key, const uint8_t *__restrict__ kp_score, int report_score,
                      float kp_size, int half, const int *__restrict__ umax, fe_kpoint *__restrict__ kp,
                      float *__restrict__ kx, float *__restrict__ ky, float2 *__restrict__ kcs) {
    const int image = blockIdx.y;
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * ORI_WARPS + (threadIdx.x >> 5);
    const int n = min((int)n_kp[image], g.kp_cap);
    if (i >= n) return;
    const size_t o = (size_t)image * g.kp_cap + i;
    const uint32_t key = kp_key[o];
    const int x = key & 0xFFFF, y = key >> 16;
    const uint8_t *src = img + (size_t)image * g.img_stride;
    int m10 = 0, m01 = 0;
    for (int v = -half; v <= half; ++v) {
        const int d = umax[v < 0 ? -v : v];
        const int yy = min(max(reflect101(y + v, g.h), 0), g.h - 1);
        int rowsum = 0;
        for (int u = -d + lane; u <= d; u += 32) {
            const int xx = min(max(reflect101(x + u, g.w), 0), g.w - 1);
            const int val = src[(size_t)yy * g.pitch + xx];
            m10 += u * val;
            rowsum += val;
        }
        m01 += v * rowsum;
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) {
        m10 += __shfl_xor_sync(0xffffffffu, m10, off);
        m01 += __shfl_xor_sync(0xffffffffu, m01, off);
    }
    if (lane == 0) {
        const float angle = fast_atan2_deg((float)m01, (float)m10);
        store_keypoint(o, key, angle, steer(angle), kp_size, kp_score, report_score, kp, kx, ky, kcs);
    }
}

// orient_pack_kernel reads the 31-px disc as aligned words straight from the image, up to 5 bytes past the disc's right end
// (they weigh 0).  Keypoints more than ORI_R px from the border keep the disc inside the image and a row of the image below
// it, so those bytes stay inside the image buffer.  Other patch sizes and nearer keypoints take orient_general_kernel.
static bool orient_fast(const DetectParams &p) { return p.patch_size == ORB_PATCH && p.edge > ORI_R; }

int launch_orient(const Geom &g, const DetectParams &p, const Buffers &b, bool orientation, cudaStream_t s) {
    const float kp_size = orientation ? (float)p.patch_size : 7.f;      // cv::ORB's keypoints are patchSize wide, cv::FAST's 7
    if (orientation && !orient_fast(p)) {       // b.umax holds OpenCV's umax table for radius patch_size / 2
        dim3 grid(div_up(g.kp_cap, ORI_WARPS), g.n_images);
        orient_general_kernel<<<grid, ORI_WARPS * 32, 0, s>>>(b.img, g, b.n_kp, b.kp_key, b.kp_score, p.nonmax ? 1 : 0, kp_size,
                                                              p.patch_size / 2, b.umax, b.kp, b.kx, b.ky, b.kcs);
        return 1;
    }
    dim3 grid(div_up(g.kp_cap, ORI_WARPS * ORI_KPW), g.n_images);
    orient_pack_kernel<<<grid, ORI_WARPS * 32, 0, s>>>(b.img, g, b.n_kp, b.kp_key, b.kp_score,
                                                       orientation ? 1 : 0, p.nonmax ? 1 : 0, kp_size,
                                                       b.kp, b.kx, b.ky, b.kcs);
    return 1;
}

// Externally supplied keypoints (fe_describe / fe_stereo_match): derive kx, ky, (cos, sin) from the
// uploaded wire-format records.  kp.angle is used literally (ORB.compute does not recompute it).
__global__ void unpack_kps_kernel(Geom g, const uint32_t *__restrict__ counts,
                                  const fe_kpoint *__restrict__ kp, float *__restrict__ kx,
                                  float *__restrict__ ky, float2 *__restrict__ kcs) {
    const int image = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= min((int)counts[image], g.kp_cap)) return;
    const size_t o = (size_t)image * g.kp_cap + i;
    const fe_kpoint k = kp[o];
    kx[o] = k.x; ky[o] = k.y;
    kcs[o] = steer(k.angle);
}

int launch_unpack_kps(const Geom &g, const Buffers &b, const uint32_t *counts, cudaStream_t s) {
    dim3 grid(div_up(g.kp_cap, 256), g.n_images);
    unpack_kps_kernel<<<grid, 256, 0, s>>>(g, counts, b.kp, b.kx, b.ky, b.kcs);
    return 1;
}

// ---- 7x7 Gaussian ----------------------------------------------------------------------------
// Tile = 128 x 32 pixels, 128 threads.  Stage 1: the raw tile (+3 halo, REFLECT_101 applied while
// staging) as bytes.  Stage 2: row pass, four pixels per thread, u8 -> f32 by the exponent trick
// (0x4B000000 | b) - 2^23 (exact, no I2F on the quarter-rate XU pipe), results as float4 in shared
// memory.  Stage 3: column pass, each thread owns one 4-pixel column group and 8 consecutive rows,
// sliding over 14 row-pass results; rounding is (s + 1.5 * 2^23) & 0xFF == rint half-even.
constexpr int BL_TW = 128, BL_TH = 32, BL_THREADS = 128;
constexpr int BL_IH = BL_TH + 6;
constexpr int BL_RAWW = BL_TW + 8;          // bytes staged per row: x0-4 .. x0+131 (34 words)

__device__ __forceinline__ float u8f(uint32_t word, int byte) {
    // float(b) = as_float(0x4B000000 | b) - 8388608.f
    const uint32_t bits = __byte_perm(word, 0x4B000000u, 0x7440 + byte);   // bytes: (b, 0, 0, 0x4B)
    return __fsub_rn(__uint_as_float(bits), 8388608.f);
}

__global__ void __launch_bounds__(BL_THREADS)
gauss7_kernel(const uint8_t *__restrict__ img, uint8_t *__restrict__ out, Geom g) {
    __shared__ __align__(16) uint8_t s_raw[BL_IH][BL_RAWW];
    __shared__ __align__(16) float4 s_row[BL_IH][BL_TW / 4];
    // getGaussianKernel(7, 2, CV_32F)
    const float g0 = 0.07015932351350784f, g1 = 0.13107487559318542f, g2 = 0.1907128244638443f,
                g3 = 0.21610593795776367f;
    const int image = blockIdx.z;
    const int x0 = blockIdx.x * BL_TW, y0 = blockIdx.y * BL_TH;
    const uint8_t *src = img + (size_t)image * g.img_stride;
    // source row of every staged row (REFLECT_101), once per tile instead of once per word
    __shared__ int s_gy[BL_IH];
    if (threadIdx.x < BL_IH) s_gy[threadIdx.x] = min(max(reflect101(y0 + (int)threadIdx.x - 3, g.h), 0), g.h - 1) * g.pitch;
    __syncthreads();
    for (int i = threadIdx.x; i < BL_IH * (BL_RAWW / 4); i += BL_THREADS) {
        const int r = i / (BL_RAWW / 4), wi = i - r * (BL_RAWW / 4);
        const uint8_t *row = src + s_gy[r];
        const int gx = x0 - 4 + 4 * wi;
        uint32_t word;
        if (gx >= 0 && gx + 3 < g.w) {
            word = __ldg(reinterpret_cast<const uint32_t *>(row + gx));
        } else {                                         // the one or two words of a row that cross the image border
            word = 0;
#pragma unroll
            for (int b = 0; b < 4; ++b)
                word |= (uint32_t)row[min(max(reflect101(gx + b, g.w), 0), g.w - 1)] << (8 * b);
        }
        *reinterpret_cast<uint32_t *>(&s_raw[r][4 * wi]) = word;
    }
    __syncthreads();
    // row pass: output pixels x0+4j .. x0+4j+3 need bytes 4j+1 .. 4j+10 of the staged row
    for (int i = threadIdx.x; i < BL_IH * (BL_TW / 4); i += BL_THREADS) {
        const int r = i / (BL_TW / 4), j = i - r * (BL_TW / 4);
        const uint32_t *wp = reinterpret_cast<const uint32_t *>(&s_raw[r][4 * j]);
        const uint32_t w0 = wp[0], w1 = wp[1], w2 = wp[2];
        float f[10];
        f[0] = u8f(w0, 1); f[1] = u8f(w0, 2); f[2] = u8f(w0, 3);
        f[3] = u8f(w1, 0); f[4] = u8f(w1, 1); f[5] = u8f(w1, 2); f[6] = u8f(w1, 3);
        f[7] = u8f(w2, 0); f[8] = u8f(w2, 1); f[9] = u8f(w2, 2);
        float o[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            float acc = __fmul_rn(f[q], g0);
            acc = __fmaf_rn(f[q + 1], g1, acc);
            acc = __fmaf_rn(f[q + 2], g2, acc);
            acc = __fmaf_rn(f[q + 3], g3, acc);
            acc = __fmaf_rn(f[q + 4], g2, acc);
            acc = __fmaf_rn(f[q + 5], g1, acc);
            acc = __fmaf_rn(f[q + 6], g0, acc);
            o[q] = acc;
        }
        s_row[r][j] = make_float4(o[0], o[1], o[2], o[3]);
    }
    __syncthreads();
    // column pass: thread = (column group j, row block of 8)
    {
        const int j = threadIdx.x & 31, rb = threadIdx.x >> 5;     // 32 groups x 4 row blocks
        const int x = x0 + 4 * j;
        float4 t[14];
#pragma unroll
        for (int k = 0; k < 14; ++k) t[k] = s_row[rb * 8 + k][j];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int y = y0 + rb * 8 + q;
            const float4 c = t[q + 3], a1 = t[q + 4], b1 = t[q + 2], a2 = t[q + 5], b2 = t[q + 1], a3 = t[q + 6], b3 = t[q];
            const float cc[4] = {c.x, c.y, c.z, c.w};
            const float p1[4] = {__fadd_rn(a1.x, b1.x), __fadd_rn(a1.y, b1.y), __fadd_rn(a1.z, b1.z), __fadd_rn(a1.w, b1.w)};
            const float p2[4] = {__fadd_rn(a2.x, b2.x), __fadd_rn(a2.y, b2.y), __fadd_rn(a2.z, b2.z), __fadd_rn(a2.w, b2.w)};
            const float p3[4] = {__fadd_rn(a3.x, b3.x), __fadd_rn(a3.y, b3.y), __fadd_rn(a3.z, b3.z), __fadd_rn(a3.w, b3.w)};
            uint32_t packed = 0;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                float acc = __fmul_rn(cc[e], g3);
                acc = __fmaf_rn(p1[e], g2, acc);
                acc = __fmaf_rn(p2[e], g1, acc);
                acc = __fmaf_rn(p3[e], g0, acc);
                // rint half-even via the 1.5 * 2^23 trick; 0 <= acc <= 255.0001
                packed |= (__float_as_uint(__fadd_rn(acc, 12582912.f)) & 0xFFu) << (8 * e);
            }
            if (y < g.h && x < g.pitch)
                *reinterpret_cast<uint32_t *>(out + (size_t)image * g.img_stride + (size_t)y * g.pitch + x) = packed;
        }
    }
}

// ---- 7x7 Gaussian, rolling form (the one launch_blur runs) -----------------------------------------------
// A warp owns a column segment of 128 pixels (lane = 4 pixels = one 32-bit word) and walks DOWN a strip of
// G7_ROWS image rows.  Per step it reads ONE image row (own word from HBM/L2, the two neighbouring words by
// lane shuffle, the segment's halo words by lanes 0 / 31), runs the row pass on it, and keeps the row-pass
// results of the last 7 rows in REGISTERS (the walk is unrolled by 7, so the window rotates by renaming);
// the column pass of the row three steps back then needs no memory at all.  No shared memory, no barrier;
// the row pass is computed once per image row (+6 halo rows per strip) instead of 38 times per 32 rows, and
// every float operation keeps OpenCV's order (SURVEY A.4): row pass s = I[x-3] g0; s = fma(I[x-3+k], gk, s);
// column pass s = T[y] g3; s = fma(T[y+k] + T[y-k], g(3-k), s); rint half-even.
constexpr int G7_ROWS = 90;                 // output rows per warp walk (6 halo rows on top: 6.7 %)
constexpr int G7_WARPS = 4;

__global__ void __launch_bounds__(G7_WARPS * 32)
gauss7_roll_kernel(const uint8_t *__restrict__ img, uint8_t *__restrict__ out, Geom g) {
    const float g0 = 0.07015932351350784f, g1 = 0.13107487559318542f, g2 = 0.1907128244638443f,
                g3 = 0.21610593795776367f;
    const int lane = threadIdx.x & 31;
    const int segm = blockIdx.x * G7_WARPS + (threadIdx.x >> 5);
    const int x0 = segm * 128;
    if (x0 >= g.w) return;                                   // whole warp
    const int image = blockIdx.z;
    const int ys = blockIdx.y * G7_ROWS, ye = min(ys + G7_ROWS, g.h);
    const uint8_t *src = img + (size_t)image * g.img_stride;
    uint8_t *dst = out + (size_t)image * g.img_stride;
    const int x = x0 + 4 * lane;                             // first of this lane's four pixels
    const uint32_t FULL = 0xffffffffu;
    // lanes whose 10-byte window x - 3 .. x + 6 leaves [0, w) assemble their three words bytewise (REFLECT_101)
    const bool fix = (x - 3 < 0) || (x + 6 >= g.w);
    const bool own_ok = x + 3 < g.pitch;                     // own word inside the padded row
    // halo words of the segment: lane 0 also loads the word left of it, lane 31 the word right of it
    const bool halo_l = lane == 0 && x0 - 4 >= 0, halo_r = lane == 31 && x0 + 131 < g.pitch;
    const int xh = halo_l ? x0 - 4 : x0 + 128;
    const bool halo = halo_l || halo_r;
    // clamped addresses: every lane always loads (no select between a load and its use two rows later)
    const uint8_t *own_p = src + min(x, g.pitch - 4), *halo_p = src + (halo ? xh : min(x, g.pitch - 4));
    auto row_off = [&](int i) { return (size_t)min(max(reflect101(ys - 3 + i, g.h), 0), g.h - 1) * (size_t)g.pitch; };

    float4 t[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) t[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    const int n_steps = ye - ys + 6;                         // staged rows ys - 3 .. ye + 2
    // two rows in flight: the words of staged rows i and i + 1 are loaded before row i is processed
    uint32_t oa = __ldg(reinterpret_cast<const uint32_t *>(own_p + row_off(0))), ha = __ldg(reinterpret_cast<const uint32_t *>(halo_p + row_off(0)));
    uint32_t ob = __ldg(reinterpret_cast<const uint32_t *>(own_p + row_off(1))), hb = __ldg(reinterpret_cast<const uint32_t *>(halo_p + row_off(1)));
    for (int base = 0; base < n_steps; base += 7) {
#pragma unroll
        for (int k = 0; k < 7; ++k) {
            const int i = base + k;                          // staged row i <-> image row ys - 3 + i
            if (i < n_steps) {
                uint32_t w1 = oa;
                const uint32_t wh = ha;
                oa = ob; ha = hb;
                {
                    const size_t ro = row_off(min(i + 2, n_steps - 1));
                    ob = __ldg(reinterpret_cast<const uint32_t *>(own_p + ro));
                    hb = __ldg(reinterpret_cast<const uint32_t *>(halo_p + ro));
                }
                uint32_t w0 = __shfl_up_sync(FULL, w1, 1), w2 = __shfl_down_sync(FULL, w1, 1);
                if (halo_l) w0 = wh;
                if (halo_r) w2 = wh;
                if (fix) {
                    const uint8_t *row = src + row_off(i);
                    w0 = w1 = w2 = 0;
#pragma unroll
                    for (int bb = 1; bb < 11; ++bb) {        // bytes 1 .. 10 of the 12-byte window = pixels x - 3 .. x + 6
                        const uint32_t pv = row[min(max(reflect101(x - 4 + bb, g.w), 0), g.w - 1)];
                        if (bb < 4) w0 |= pv << (8 * bb);
                        else if (bb < 8) w1 |= pv << (8 * (bb - 4));
                        else w2 |= pv << (8 * (bb - 8));
                    }
                }
                float f[10];
                f[0] = u8f(w0, 1); f[1] = u8f(w0, 2); f[2] = u8f(w0, 3);
                f[3] = u8f(w1, 0); f[4] = u8f(w1, 1); f[5] = u8f(w1, 2); f[6] = u8f(w1, 3);
                f[7] = u8f(w2, 0); f[8] = u8f(w2, 1); f[9] = u8f(w2, 2);
                float o[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    float acc = __fmul_rn(f[q], g0);
                    acc = __fmaf_rn(f[q + 1], g1, acc);
                    acc = __fmaf_rn(f[q + 2], g2, acc);
                    acc = __fmaf_rn(f[q + 3], g3, acc);
                    acc = __fmaf_rn(f[q + 4], g2, acc);
                    acc = __fmaf_rn(f[q + 5], g1, acc);
                    acc = __fmaf_rn(f[q + 6], g0, acc);
                    o[q] = acc;
                }
                t[k] = make_float4(o[0], o[1], o[2], o[3]);
                if (i >= 6) {
                    // output row = staged row i - 3; rows i - 6 .. i are t[(k + 1) % 7] .. t[k]
                    const float4 c = t[(k + 4) % 7], a1 = t[(k + 5) % 7], b1 = t[(k + 3) % 7], a2 = t[(k + 6) % 7], b2 = t[(k + 2) % 7],
                                 a3 = t[k], b3 = t[(k + 1) % 7];
                    const float cc[4] = {c.x, c.y, c.z, c.w};
                    const float p1[4] = {__fadd_rn(a1.x, b1.x), __fadd_rn(a1.y, b1.y), __fadd_rn(a1.z, b1.z), __fadd_rn(a1.w, b1.w)};
                    const float p2[4] = {__fadd_rn(a2.x, b2.x), __fadd_rn(a2.y, b2.y), __fadd_rn(a2.z, b2.z), __fadd_rn(a2.w, b2.w)};
                    const float p3[4] = {__fadd_rn(a3.x, b3.x), __fadd_rn(a3.y, b3.y), __fadd_rn(a3.z, b3.z), __fadd_rn(a3.w, b3.w)};
                    uint32_t rb[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        float acc = __fmul_rn(cc[e], g3);
                        acc = __fmaf_rn(p1[e], g2, acc);
                        acc = __fmaf_rn(p2[e], g1, acc);
                        acc = __fmaf_rn(p3[e], g0, acc);
                        rb[e] = __float_as_uint(__fadd_rn(acc, 12582912.f));   // rint half-even in the low mantissa byte; 0 <= acc <= 255.0001
                    }
                    const uint32_t packed = __byte_perm(__byte_perm(rb[0], rb[1], 0x0040), __byte_perm(rb[2], rb[3], 0x0040), 0x5410);
                    const int y = ys + i - 6;
                    if (own_ok) *reinterpret_cast<uint32_t *>(dst + (size_t)y * g.pitch + x) = packed;
                }
            }
        }
    }
}

int launch_blur(const Geom &g, const Buffers &b, cudaStream_t s) {
    dim3 grid(div_up(div_up(g.w, 128), G7_WARPS), div_up(g.h, G7_ROWS), g.n_images);
    gauss7_roll_kernel<<<grid, G7_WARPS * 32, 0, s>>>(b.img, b.blur, g);
    return 1;
}

// ---- rBRIEF-256 ------------------------------------------------------------------------------
constexpr int BR_WARPS = 8;
constexpr int BR_KPW = 8;                   // keypoints per warp (amortises the pattern copy)
constexpr int BR_R = 19;                    // |rotated pattern offset| <= rint(18.39) -> 19 is safe
constexpr int BR_ROWS = 2 * BR_R + 1;       // 39
constexpr int BR_WORDS = 11;                // 39 + 3 alignment bytes -> 11 words per row
constexpr int BR_STRIDE = 12;               // words per patch row in shared memory

// rint (half-even) of |v| < 2^22 without the quarter-rate F2I: the FADD against 1.5 * 2^23 rounds to the nearest
// even integer exactly like cvRound / __float2int_rn, and the integer sits in the low mantissa bits.
__device__ __forceinline__ int rint_small(float v) {
    return __float_as_int(__fadd_rn(v, 12582912.f)) - 0x4B400000;
}

// pattern point (x, y) steered by (a, b) = (cos, sin): orb.cpp's GET_VALUE in f32, without FMA
__device__ __forceinline__ float2 steer_point(float x, float y, float a, float b) {
    return make_float2(__fsub_rn(__fmul_rn(x, a), __fmul_rn(y, b)), __fadd_rn(__fmul_rn(x, b), __fmul_rn(y, a)));
}

// Lane l always evaluates tests l, l + 32, ..., l + 224: its eight point pairs of bit_pattern_31_ live in registers as f32 for
// all the keypoints it describes (no I2F and no shared-memory pattern reads in the test loop -- the LSU pipe bounds it)
__device__ __forceinline__ void load_pattern(float4 (&pat)[8], int lane) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const char4 pt = reinterpret_cast<const char4 *>(d_pattern)[j * 32 + lane];
        pat[j] = make_float4((float)pt.x, (float)pt.y, (float)pt.z, (float)pt.w);
    }
}

// The 256 tests of one keypoint steered by (a, b) on a blurred patch in shared memory with rows ROW_BYTES apart; `centre` is
// the shared-memory address of the keypoint's pixel.  The ballot of test j * 32 + l is exactly little-endian word j of the
// 32-byte descriptor (bit i of byte b <-> test 8b + i): returned in lane j (lanes 0-7).
template <int ROW_BYTES>
__device__ __forceinline__ uint32_t rbrief_tests(const float4 (&pat)[8], float a, float b, uint32_t centre, int lane) {
    // rint_small() leaves 0x4B400000 + i in the float's bits: the address of sample (ix, iy) is then
    //   centre + iy * ROW_BYTES + ix = (centre - (ROW_BYTES + 1) * 0x4B400000) + bits_y * ROW_BYTES + bits_x   (32-bit wrap-around)
    const uint32_t base = centre - 0x4B400000u * (uint32_t)(ROW_BYTES + 1);
    auto sample = [&](float px, float py) {      // blurred pixel at (rint, rint) of the steered point
        const float2 r = steer_point(px, py, a, b);
        const uint32_t bx = __float_as_uint(__fadd_rn(r.x, 12582912.f)), by = __float_as_uint(__fadd_rn(r.y, 12582912.f));
        uint32_t v;
        asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(base + by * (uint32_t)ROW_BYTES + bx));
        return v;
    };
    uint32_t word = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const uint32_t t0 = sample(pat[j].x, pat[j].y);
        const uint32_t t1 = sample(pat[j].z, pat[j].w);
        const uint32_t w = __ballot_sync(0xffffffffu, t0 < t1);
        if (lane == j) word = w;
    }
    return word;
}

// One warp per keypoint.  The 39 x 39 neighbourhood of the blurred image is first staged in shared
// memory with aligned 32-bit loads (rows coalesced: ~80 sectors per keypoint instead of 512 scattered
// byte gathers from L1), then the 256 tests sample the staged patch.
__global__ void __launch_bounds__(BR_WARPS * 32)
rbrief_kernel(const uint8_t *__restrict__ blur, Geom g, const uint32_t *__restrict__ counts,
              const float *__restrict__ kx, const float *__restrict__ ky,
              const float2 *__restrict__ kcs, uint8_t *__restrict__ desc) {
    __shared__ uint32_t s_patch[BR_WARPS][BR_ROWS * BR_STRIDE];
    const int image = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = min((int)counts[image], g.kp_cap);
    if (blockIdx.x * (BR_WARPS * BR_KPW) >= n) return;
    float4 pat[8];
    load_pattern(pat, lane);
    uint32_t *patch = s_patch[warp];
    // lane `it` fetches the record of the warp's keypoint `it` up front: one load latency per warp, not per keypoint
    float pre_x = 0.f, pre_y = 0.f;
    float2 pre_cs = make_float2(1.f, 0.f);
    {
        const int i = (blockIdx.x * BR_KPW + lane) * BR_WARPS + warp;
        if (lane < BR_KPW && i < n) {
            const size_t o = (size_t)image * g.kp_cap + i;
            pre_x = kx[o]; pre_y = ky[o]; pre_cs = kcs[o];
        }
    }
    // staging geometry of this lane, the same for every keypoint: three patch rows per round (lanes 0-10, 11-21, 22-31 take
    // words 0-10, 0-10, 0-9 of rows r0, r0+1, r0+2), one more round for the eleventh word of the third rows
    const int st_w = lane % BR_WORDS, st_r = lane / BR_WORDS;
    const int st_goff = st_r * g.pitch + 4 * st_w, st_soff = st_r * BR_STRIDE + st_w;
    const int st_xoff = (3 * lane + 2) * g.pitch + 4 * (BR_WORDS - 1), st_xs = (3 * lane + 2) * BR_STRIDE + BR_WORDS - 1;
#pragma unroll 1
    for (int it = 0; it < BR_KPW; ++it) {
    const int i = (blockIdx.x * BR_KPW + it) * BR_WARPS + warp;
    if (i >= n) break;
    const size_t o = (size_t)image * g.kp_cap + i;
    const int cx = __float2int_rn(__shfl_sync(0xffffffffu, pre_x, it)), cy = __float2int_rn(__shfl_sync(0xffffffffu, pre_y, it));
    const float a = __shfl_sync(0xffffffffu, pre_cs.x, it), b = __shfl_sync(0xffffffffu, pre_cs.y, it);
    const int xl = cx - BR_R, xa = xl & ~3, off = xl - xa;
    const uint8_t *base = blur + (size_t)image * g.img_stride + (size_t)(cy - BR_R) * g.pitch + xa;
    __syncwarp();
    {
        const uint8_t *gp = base + st_goff;
        uint32_t *sp = patch + st_soff;
#pragma unroll
        for (int r0 = 0; r0 < BR_ROWS; r0 += 3) {
            *sp = __ldg(reinterpret_cast<const uint32_t *>(gp));
            gp += 3 * g.pitch; sp += 3 * BR_STRIDE;
        }
        if (lane < BR_ROWS / 3) patch[st_xs] = __ldg(reinterpret_cast<const uint32_t *>(base + st_xoff));
    }
    __syncwarp();
    const uint8_t *pc = reinterpret_cast<const uint8_t *>(patch) + BR_R * (BR_STRIDE * 4) + BR_R + off;  // centre
    const uint32_t word = rbrief_tests<BR_STRIDE * 4>(pat, a, b, (uint32_t)__cvta_generic_to_shared(pc), lane);
    if (lane < 8) reinterpret_cast<uint32_t *>(desc + o * 32)[lane] = word;
    }
}

// ---- orientation + rBRIEF per image tile ---------------------------------------------------------------------------------
// Detect-and-describe of the default geometry (describe_tile_fits, FAST score, one level): one CTA per (image, DT_ROWS x
// DT_COLS tile of keypoint centres).  The CTA stages the raw and the blurred tile with a 19-px halo in shared memory once and
// describes every keypoint of the tile from there.  orient_pack_kernel + rbrief_kernel instead re-read each keypoint's
// neighbourhood from global memory: at ~5 200 keypoints per 1280 x 720 image that is ~15x the image, the tiles stage ~2x it
// (halo included).  Keypoints are in raster order (kp_key ascending y << 16 | x per image), so those of the tile's rows are one
// index range, found by binary search.  Moments, angle, steering and the 256 tests are the helpers orient_pack_kernel and
// rbrief_kernel call: the outputs are bit-identical.
constexpr int DT_ROWS = 64, DT_COLS = 256;          // 64 x 128 and 32 x 256 tiles measured slower (more CTAs and halo)
constexpr int DT_TROWS = DT_ROWS + 2 * BR_R;                // staged rows y0 - 19 .. y0 + DT_ROWS + 18
// staged columns x0 - 32 .. x0 + DT_COLS + 31: 16-byte aligned (x0 is), they cover the reach -19 .. +20 of a keypoint (the
// orientation's 9th word ends at x + 20; those bytes weigh 0 but are read)
constexpr int DT_XL = 32;
constexpr int DT_VECS = (DT_COLS + 2 * DT_XL) / 16;         // 16-byte vectors per staged row
// raw-tile row pitch in words: 105 == 9 mod 32, so the 32 consecutive (row, word) slots of a 31 x 9-word patch read by a warp
// fall on 32 distinct banks; blurred-tile row pitch 336 bytes: 16-byte rows, and 84 words == -12 mod 32 spreads the rotated
// samples over the banks as rbrief_kernel's 12-word patch rows do
constexpr int DT_RAW_W = 105;
constexpr int DT_BLUR_B = 336;
constexpr int DT_WARPS = 8, DT_THREADS = DT_WARPS * 32;
constexpr int DT_CHUNK = 2 * DT_THREADS;                               // indices of the tile's row band examined per pass
constexpr int DT_STAGE = (2 * DT_TROWS * DT_VECS + DT_THREADS - 1) / DT_THREADS;   // 16-byte loads per thread
constexpr int DT_SMEM = DT_TROWS * DT_BLUR_B + DT_TROWS * DT_RAW_W * 4;             // dynamic: the two tiles
static_assert(DT_COLS % 16 == 0 && DT_XL % 16 == 0 && DT_XL >= BR_R, "staged columns must start 16-byte aligned");
static_assert(DT_VECS * 16 <= DT_BLUR_B && DT_VECS * 4 <= DT_RAW_W && DT_BLUR_B % 16 == 0, "staged row fits the tile row");
static_assert(DT_COLS + 2 * DT_XL - DT_XL >= DT_COLS + 21, "right halo reaches x + 20");
static_assert(DT_RAW_W % 32 == 9 && (DT_BLUR_B / 4) % 32 == 20, "bank spread of the tile rows");

__global__ void __launch_bounds__(DT_THREADS, 2)
orb_describe_tile_kernel(const uint8_t *__restrict__ img, const uint8_t *__restrict__ blur, Geom g,
                         const uint32_t *__restrict__ n_kp, const uint32_t *__restrict__ kp_key,
                         const uint8_t *__restrict__ kp_score, int report_score, float kp_size, fe_kpoint *__restrict__ kp,
                         float *__restrict__ kx, float *__restrict__ ky, float2 *__restrict__ kcs, uint8_t *__restrict__ desc) {
    extern __shared__ __align__(16) uint8_t s_blur[];                                // [DT_TROWS][DT_BLUR_B]
    uint32_t *s_raw = reinterpret_cast<uint32_t *>(s_blur + DT_TROWS * DT_BLUR_B);   // [DT_TROWS][DT_RAW_W]
    __shared__ uint32_t s_idx[DT_CHUNK], s_key[DT_CHUNK];
    __shared__ int s_range[2], s_cnt;
    const uint32_t FULL = 0xffffffffu;
    const int image = blockIdx.z;
    const int x0 = blockIdx.x * DT_COLS, y0 = blockIdx.y * DT_ROWS;
    const int ty0 = y0 - BR_R, sx = x0 - DT_XL;                 // image coordinates of tile row 0 / tile byte 0
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // both tiles, clipped to the image rows and the row pitch (what lies outside is never sampled: keypoints are >= 19 px
    // inside the image).  The loads are issued first: their latency overlaps the keypoint search.
    uint4 v[DT_STAGE];
#pragma unroll
    for (int k = 0; k < DT_STAGE; ++k) {
        const int i = threadIdx.x + k * DT_THREADS;
        const int t = i >= DT_TROWS * DT_VECS;                      // 0: blurred tile, 1: raw tile
        const int j = i - t * DT_TROWS * DT_VECS, r = j / DT_VECS, c = sx + 16 * (j - r * DT_VECS), gy = ty0 + r;
        v[k] = make_uint4(0u, 0u, 0u, 0u);
        if (i < 2 * DT_TROWS * DT_VECS && gy >= 0 && gy < g.h && c >= 0 && c < g.pitch)
            v[k] = __ldg(reinterpret_cast<const uint4 *>((t ? img : blur) + (size_t)image * g.img_stride + (size_t)gy * g.pitch + c));
    }
    const int n = min((int)n_kp[image], g.kp_cap);
    const uint32_t *keys = kp_key + (size_t)image * g.kp_cap;
    if (warp < 2) {                                             // the keypoints of rows y0 .. y0 + DT_ROWS - 1
        const int r = warp_lower_bound(keys, n, (uint32_t)(y0 + warp * DT_ROWS) << 16, lane);
        if (lane == 0) s_range[warp] = r;
    }
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    const int lo = s_range[0], hi = s_range[1];
    if (lo >= hi) return;
#pragma unroll
    for (int k = 0; k < DT_STAGE; ++k) {
        const int i = threadIdx.x + k * DT_THREADS;
        if (i >= 2 * DT_TROWS * DT_VECS) break;
        const int t = i >= DT_TROWS * DT_VECS;
        const int j = i - t * DT_TROWS * DT_VECS, r = j / DT_VECS, q = j - r * DT_VECS;
        if (t == 0) {
            *reinterpret_cast<uint4 *>(s_blur + r * DT_BLUR_B + 16 * q) = v[k];
        } else {
            uint32_t *d = s_raw + r * DT_RAW_W + 4 * q;
            d[0] = v[k].x; d[1] = v[k].y; d[2] = v[k].z; d[3] = v[k].w;
        }
    }
    int soff[ORI_K], sv[ORI_K];                 // the orientation's slot geometry in raw-tile words
    ori_slots(lane, DT_RAW_W, 1, soff, sv);
    float4 pat[8];
    load_pattern(pat, lane);
    // shared-memory address of image pixel (0, 0) in the blurred tile's coordinates
    const uint32_t blur_o = (uint32_t)__cvta_generic_to_shared(s_blur) - (uint32_t)(ty0 * DT_BLUR_B + sx);
    for (int base = lo; base < hi; base += DT_CHUNK) {
        // the band's keypoints whose x lies in the tile (any order: every result goes to its keypoint's own index).  This is
        // tile_collect (fe_internal.cuh, which brief_tile_kernel calls) written out: through the helper this kernel compiles
        // to 1960 instead of 1880 instructions, and c2 ran 41.40 k against 41.69 k pairs/s (profiles/r7_ab_brief.log)
#pragma unroll
        for (int q = 0; q < DT_CHUNK / DT_THREADS; ++q) {
            const int i = base + q * DT_THREADS + (int)threadIdx.x;
            uint32_t key = 0;
            bool in = false;
            if (i < hi) {
                key = keys[i];
                in = (int)(key & 0xFFFF) >= x0 && (int)(key & 0xFFFF) < x0 + DT_COLS;
            }
            const uint32_t m = __ballot_sync(FULL, in);
            int pos = 0;
            if (lane == 0 && m) pos = atomicAdd(&s_cnt, __popc(m));
            pos = __shfl_sync(FULL, pos, 0) + __popc(m & ((1u << lane) - 1u));
            if (in) { s_idx[pos] = (uint32_t)i; s_key[pos] = key; }
        }
        __syncthreads();                                        // (also: the tiles are staged)
        const int m = s_cnt;
        __syncthreads();
        if (threadIdx.x == 0) s_cnt = 0;
        // warp w takes list entries w, w + 8, ...: lane j holds entry w + 8 j of each group of 256
        for (int grp = 0; grp < m; grp += DT_THREADS) {
            const int e = grp + warp + DT_WARPS * lane;
            const bool valid = e < m;
            const int cnt = __popc(__ballot_sync(FULL, valid));
            if (cnt == 0) break;
            const uint32_t my_key = valid ? s_key[e] : 0u;
            const int my_i = valid ? (int)s_idx[e] : 0;
            float my_angle = 0.f;
            // intensity-centroid orientation, two keypoints per round (orient_pack_kernel)
#pragma unroll 1
            for (int it = 0; it < cnt; it += 2) {
                const bool two = it + 1 < cnt;
                const uint32_t key0 = __shfl_sync(FULL, my_key, it), key1 = __shfl_sync(FULL, my_key, two ? it + 1 : it);
                const int xl0 = (int)(key0 & 0xFFFF) - ORI_R, xa0 = xl0 & ~3;
                const int xl1 = (int)(key1 & 0xFFFF) - ORI_R, xa1 = xl1 & ~3;
                const uint32_t *p0 = s_raw + ((int)(key0 >> 16) - ORI_R - ty0) * DT_RAW_W + ((xa0 - sx) >> 2);
                const uint32_t *p1 = s_raw + ((int)(key1 >> 16) - ORI_R - ty0) * DT_RAW_W + ((xa1 - sx) >> 2);
                auto words = [&](int k) {
                    const bool in = lane + 32 * k < ORI_SLOTS;
                    return make_uint2(in ? p0[soff[k]] : 0u, in ? p1[soff[k]] : 0u);
                };
                const float2 angles = ori_angles(words, xl0 - xa0, xl1 - xa1, d_ori_tab.u, d_ori_tab.m, sv, lane);
                if (lane == it) my_angle = angles.x;
                if (two && lane == it + 1) my_angle = angles.y;
            }
            // the record and the steering, every lane its own keypoint
            float2 cs = make_float2(1.f, 0.f);
            if (valid) {
                cs = steer(my_angle);
                store_keypoint((size_t)image * g.kp_cap + my_i, my_key, my_angle, cs, kp_size, kp_score, report_score,
                               kp, kx, ky, kcs);
            }
            // rBRIEF-256 from the blurred tile (rbrief_kernel)
#pragma unroll 1
            for (int it = 0; it < cnt; ++it) {
                const uint32_t key = __shfl_sync(FULL, my_key, it);
                const int i = __shfl_sync(FULL, my_i, it);
                const float a = __shfl_sync(FULL, cs.x, it), b = __shfl_sync(FULL, cs.y, it);
                const uint32_t word = rbrief_tests<DT_BLUR_B>(pat, a, b, blur_o + (key >> 16) * (uint32_t)DT_BLUR_B + (key & 0xFFFF), lane);
                if (lane < 8) reinterpret_cast<uint32_t *>(desc + ((size_t)image * g.kp_cap + i) * 32)[lane] = word;
            }
        }
        __syncthreads();                                        // the list is rewritten by the next pass
    }
}

// rbrief_kernel stages the blurred image within BR_R px of each keypoint without a border, and orb_describe_tile_kernel stages
// image tiles the same way: both serve bit_pattern_31_ (WTA_K 2) at keypoints at least BR_R px from the border.
static bool rbrief_fast(const DetectParams &p) { return p.wta_k == 2 && p.patch_size == ORB_PATCH && p.edge >= BR_R; }

bool describe_tile_fits(const DetectParams &p) { return orient_fast(p) && rbrief_fast(p); }

int launch_describe_tile(const Geom &g, const DetectParams &p, const Buffers &b, cudaStream_t s) {
    static bool smem_set[64] = {false};         // per device: the attribute belongs to the device's context
    int dev = 0;
    cudaGetDevice(&dev);
    if (!smem_set[dev & 63]) {
        cudaFuncSetAttribute(orb_describe_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DT_SMEM);
        smem_set[dev & 63] = true;
    }
    dim3 grid(div_up(g.w, DT_COLS), div_up(g.h, DT_ROWS), g.n_images);
    orb_describe_tile_kernel<<<grid, DT_THREADS, DT_SMEM, s>>>(b.img, b.blur, g, b.n_kp, b.kp_key, b.kp_score, p.nonmax ? 1 : 0,
                                                               (float)p.patch_size, b.kp, b.kx, b.ky, b.kcs, b.desc);
    return 1;
}

// Sample of cv::ORB's bordered image at the keypoint (cx, cy) plus the steered, rounded pattern point (px, py): the blurred
// pixel inside the image; outside it the RAW pixel at the BORDER_REFLECT_101 position, because cv2 blurs only the image area
// of its bordered buffer (pinned against cv2 4.13 with patchSize 70, where 8.7 % of the descriptors touch the border)
__device__ __forceinline__ int bordered_sample(const uint8_t *bl, const uint8_t *rw, const Geom &g, int cx, int cy, float px,
                                               float py, float a, float b) {
    const float2 r = steer_point(px, py, a, b);
    int x = cx + rint_small(r.x), y = cy + rint_small(r.y);
    if (x >= 0 && x < g.w && y >= 0 && y < g.h) return bl[(size_t)y * g.pitch + x];
    x = min(max(reflect101(x, g.w), 0), g.w - 1);
    y = min(max(reflect101(y, g.h), 0), g.h - 1);
    return rw[(size_t)y * g.pitch + x];
}

// rBRIEF-256 with a caller-selected pattern (ORB::setPatchSize != 31 -> makeRandomPattern, bin/detect_node:50-51), or the
// built-in one at keypoints nearer the border than BR_R.  No staging: the pattern may reach half_patch * sqrt(2) px.
__global__ void __launch_bounds__(BR_WARPS * 32)
rbrief_general_kernel(const uint8_t *__restrict__ blur, const uint8_t *__restrict__ raw, Geom g,
                      const uint32_t *__restrict__ counts, const float *__restrict__ kx, const float *__restrict__ ky,
                      const float2 *__restrict__ kcs, const int8_t *__restrict__ pattern, uint8_t *__restrict__ desc) {
    __shared__ float4 s_pat[256];
    for (int i = threadIdx.x; i < 256; i += BR_WARPS * 32) {
        const char4 pt = reinterpret_cast<const char4 *>(pattern)[i];
        s_pat[i] = make_float4((float)pt.x, (float)pt.y, (float)pt.z, (float)pt.w);
    }
    __syncthreads();
    const int image = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = min((int)counts[image], g.kp_cap);
    const int i = blockIdx.x * BR_WARPS + warp;
    if (i >= n) return;
    const size_t o = (size_t)image * g.kp_cap + i;
    const int cx = __float2int_rn(kx[o]), cy = __float2int_rn(ky[o]);
    const float2 cs = kcs[o];
    const uint8_t *bl = blur + (size_t)image * g.img_stride, *rw = raw + (size_t)image * g.img_stride;
    uint32_t word = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float4 pt = s_pat[j * 32 + lane];
        const int t0 = bordered_sample(bl, rw, g, cx, cy, pt.x, pt.y, cs.x, cs.y);
        const int t1 = bordered_sample(bl, rw, g, cx, cy, pt.z, pt.w, cs.x, cs.y);
        const uint32_t w = __ballot_sync(0xffffffffu, t0 < t1);
        if (lane == j) word = w;
    }
    if (lane < 8) reinterpret_cast<uint32_t *>(desc + o * 32)[lane] = word;
}

// ORB with WTA_K = 3 / 4 (orb.cpp computeOrbDescriptors): 128 tuples of K points, two bits per tuple = index of the
// largest sample (K = 3: t2 > t1 ? (t2 > t0 ? 2 : 0) : (t1 > t0);  K = 4: winner of (t0 | t1) vs winner of (t2 | t3),
// ties resolved exactly as OpenCV's strict comparisons do).  Lane l computes byte l (tuples 4l .. 4l + 3).
template <int K>
__global__ void __launch_bounds__(BR_WARPS * 32)
rbrief_wta_kernel(const uint8_t *__restrict__ blur, const uint8_t *__restrict__ raw, Geom g,
                  const uint32_t *__restrict__ counts, const float *__restrict__ kx, const float *__restrict__ ky,
                  const float2 *__restrict__ kcs, const int8_t *__restrict__ pattern, uint8_t *__restrict__ desc) {
    __shared__ float2 s_pat[512];
    for (int i = threadIdx.x; i < 128 * K; i += BR_WARPS * 32) s_pat[i] = make_float2((float)pattern[2 * i], (float)pattern[2 * i + 1]);
    __syncthreads();
    const int image = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = min((int)counts[image], g.kp_cap);
    const int i = blockIdx.x * BR_WARPS + warp;
    if (i >= n) return;
    const size_t o = (size_t)image * g.kp_cap + i;
    const int cx = __float2int_rn(kx[o]), cy = __float2int_rn(ky[o]);
    const float2 cs = kcs[o];
    const uint8_t *bl = blur + (size_t)image * g.img_stride, *rw = raw + (size_t)image * g.img_stride;
    auto sample = [&](int idx) { return bordered_sample(bl, rw, g, cx, cy, s_pat[idx].x, s_pat[idx].y, cs.x, cs.y); };
    uint32_t val = 0;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const int base = (lane * 4 + t) * K;
        int k;
        if (K == 3) {
            const int t0 = sample(base), t1 = sample(base + 1), t2 = sample(base + 2);
            k = t2 > t1 ? (t2 > t0 ? 2 : 0) : (t1 > t0 ? 1 : 0);
        } else {
            int t0 = sample(base), t2 = sample(base + 2);
            const int t1 = sample(base + 1), t3 = sample(base + 3);
            int u = 0, v = 2;
            if (t1 > t0) { t0 = t1; u = 1; }
            if (t3 > t2) { t2 = t3; v = 3; }
            k = t0 > t2 ? u : v;
        }
        val |= (uint32_t)k << (2 * t);
    }
    desc[o * 32 + lane] = (uint8_t)val;
}

int launch_rbrief(const Geom &g, const DetectParams &p, const Buffers &b, const uint32_t *counts, cudaStream_t s) {
    if (rbrief_fast(p)) {
        dim3 grid(div_up(g.kp_cap, BR_WARPS * BR_KPW), g.n_images);
        rbrief_kernel<<<grid, BR_WARPS * 32, 0, s>>>(b.blur, g, counts, b.kx, b.ky, b.kcs, b.desc);
        return 1;
    }
    // b.pattern holds the ctx's pattern (bit_pattern_31_ or makeRandomPattern(patch_size)), as WTA_K-point tuples for WTA_K 3 / 4
    dim3 grid(div_up(g.kp_cap, BR_WARPS), g.n_images);
    if (p.wta_k == 3) rbrief_wta_kernel<3><<<grid, BR_WARPS * 32, 0, s>>>(b.blur, b.img, g, counts, b.kx, b.ky, b.kcs, b.pattern, b.desc);
    else if (p.wta_k == 4) rbrief_wta_kernel<4><<<grid, BR_WARPS * 32, 0, s>>>(b.blur, b.img, g, counts, b.kx, b.ky, b.kcs, b.pattern, b.desc);
    else rbrief_general_kernel<<<grid, BR_WARPS * 32, 0, s>>>(b.blur, b.img, g, counts, b.kx, b.ky, b.kcs, b.pattern, b.desc);
    return 1;
}

}  // namespace fe
