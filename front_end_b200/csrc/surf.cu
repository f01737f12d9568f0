// SURF / SURF_EXTENDED descriptor extraction at provided keypoints.
//
// Replaces cv::SURF::operator()(img, mask, keypoints, descriptors, useProvidedKeypoints = true) of
// the reference's vendored OpenCV-2.4 nonfree module -- /root/reference src/surf.cpp:896-980 (driver)
// and SURFInvoker::operator() :563-851 -- as selected by getDescriptor("SURF")
// (src/front_end/features.py:455-457) and bin/detect_node:33-41 (extended + upright on FAST keypoints).
//
// One warp per keypoint.  Every float operation is written in the reference's order with explicit
// non-fused intrinsics (the library is built with -fmad=false): orientation samples keep their index
// order when compacted, sliding-window sums and cell sums are sequential per accumulator, square_mag is
// one sequential double sum.  The u8 quantisation points (window sample cvRound, INTER_AREA patch) are
// reproduced exactly, including OpenCV's three INTER_AREA code paths: the general area table for
// win_size > 21, integer box sums when win_size is a multiple of 21 (ResizeAreaFast) and, for
// win_size < 21 (FAST keypoints, size 7 -> win 19), the fall-back to bilinear with area-mode
// coefficients in 2^11 fixed point.
#include <cmath>
#include <mutex>

#include "fe_internal.cuh"

namespace fe {

constexpr int S_WARPS_SMALL = 8, S_WARPS_LARGE = 4;      // warps per CTA for the 32-px / 88-px window variants
constexpr int PATCH = 20;           // PATCH_SZ
constexpr int PW = PATCH + 1;       // 21
constexpr int ORI_RADIUS = SURF_ORI_RADIUS, N_ORI = 113;

__device__ float d_aptw[N_ORI];     // Gaussian weights of the orientation samples (sigma 2.5)
__device__ int8_t d_apt[N_ORI][2];  // sample offsets (x, y)
__device__ float d_dw[PATCH * PATCH];   // descriptor weights (sigma 3.3), plain-formula Gaussian
// resize(win, 21 x 21, INTER_AREA) of a window SMALLER than 21 px is OpenCV's bilinear path with area-mode coefficients
// (INTER_RESIZE_COEF_BITS = 11): source index and the two 11-bit weights of destination index d, for every S in 1 .. 20
struct UpCoef { int sx, a0, a1; };
__device__ UpCoef d_up[PW][PW];         // [S][d]

static void upload_tables() {
    static std::once_flag once[64];     // the tables are per-device symbols
    int dev = 0;
    cudaGetDevice(&dev);
    std::call_once(once[dev & 63], [] {
        auto gauss = [](int n, double sigma, float *out) {
            // OpenCV 2.4 getGaussianKernel(n, sigma, CV_32F) for n without a fixed table
            const double scale2x = -0.5 / (sigma * sigma);
            double sum = 0;
            for (int i = 0; i < n; ++i) {
                const double x = i - (n - 1) * 0.5;
                out[i] = (float)std::exp(scale2x * x * x);
                sum += out[i];
            }
            sum = 1. / sum;
            for (int i = 0; i < n; ++i) out[i] = (float)(out[i] * sum);
        };
        float g_ori[2 * ORI_RADIUS + 1], g_desc[PATCH];
        gauss(2 * ORI_RADIUS + 1, 2.5, g_ori);
        gauss(PATCH, 3.3, g_desc);
        float aptw[N_ORI];
        int8_t apt[N_ORI][2];
        int n = 0;
        for (int i = -ORI_RADIUS; i <= ORI_RADIUS; ++i)
            for (int j = -ORI_RADIUS; j <= ORI_RADIUS; ++j)
                if (i * i + j * j <= ORI_RADIUS * ORI_RADIUS) {
                    apt[n][0] = (int8_t)i; apt[n][1] = (int8_t)j;
                    aptw[n++] = g_ori[i + ORI_RADIUS] * g_ori[j + ORI_RADIUS];
                }
        float dw[PATCH * PATCH];
        for (int i = 0; i < PATCH; ++i)
            for (int j = 0; j < PATCH; ++j) dw[i * PATCH + j] = g_desc[i] * g_desc[j];
        cudaMemcpyToSymbol(d_aptw, aptw, sizeof(aptw));
        cudaMemcpyToSymbol(d_apt, apt, sizeof(apt));
        cudaMemcpyToSymbol(d_dw, dw, sizeof(dw));
        static UpCoef up[PW][PW];
        for (int S = 1; S < PW; ++S)
            for (int d = 0; d < PW; ++d) {
                const double scale = (double)S / PW, inv = (double)PW / S;
                int sx = (int)std::floor(d * scale);
                float fx = (float)((d + 1) - (sx + 1) * inv);
                fx = fx <= 0.f ? 0.f : fx - std::floor(fx);
                if (sx < 0) { fx = 0.f; sx = 0; }
                if (sx >= S - 1) { fx = 0.f; sx = S - 1; }
                up[S][d].sx = sx;
                up[S][d].a0 = (int)std::lrintf((1.f - fx) * 2048.f);
                up[S][d].a1 = (int)std::lrintf(fx * 2048.f);
            }
        cudaMemcpyToSymbol(d_up, up, sizeof(up));
    });
}

// ---- integral image (cv::integral, CV_32S): (h+1) x (w+1), S[y+1][x+1] = sum of img[0..y][0..x] ------
__global__ void integral_rows_kernel(const uint8_t *__restrict__ img, int32_t *__restrict__ integ, Geom g) {
    // one warp per image row: running prefix in chunks of 32 pixels
    const int image = blockIdx.y;
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= g.h) return;
    const uint8_t *src = img + (size_t)image * g.img_stride + (size_t)row * g.pitch;
    int32_t *dst = integ + ((size_t)image * (g.h + 1) + row + 1) * (g.w + 1);
    if (lane == 0) dst[0] = 0;
    int carry = 0;
    for (int x0 = 0; x0 < g.w; x0 += 32) {
        const int x = x0 + lane;
        int v = x < g.w ? src[x] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int n = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o) v += n;
        }
        if (x < g.w) dst[x + 1] = carry + v;
        carry += __shfl_sync(0xffffffffu, v, 31);
    }
}

__global__ void integral_cols_kernel(int32_t *__restrict__ integ, Geom g) {
    const int image = blockIdx.y;
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x > g.w) return;
    int32_t *p = integ + (size_t)image * (g.h + 1) * (g.w + 1) + x;
    int acc = 0;
    p[0] = 0;
    for (int y = 1; y <= g.h; ++y) {
        acc += p[(size_t)y * (g.w + 1)];
        p[(size_t)y * (g.w + 1)] = acc;
    }
}

// ---- helpers ---------------------------------------------------------------------------------------------
struct HaarBox { int dx1, dy1, dx2, dy2; float w; };

// resizeHaarPattern (src/surf.cpp:136-152) for one box of the 4-wide pattern
__device__ __forceinline__ HaarBox haar_box(int a, int b, int c, int d, int wgt, int new_size) {
    const float ratio = __fdiv_rn((float)new_size, 4.f);
    HaarBox h;
    h.dx1 = __float2int_rn(__fmul_rn(ratio, (float)a));
    h.dy1 = __float2int_rn(__fmul_rn(ratio, (float)b));
    h.dx2 = __float2int_rn(__fmul_rn(ratio, (float)c));
    h.dy2 = __float2int_rn(__fmul_rn(ratio, (float)d));
    h.w = __fdiv_rn((float)wgt, __fmul_rn((float)(h.dx2 - h.dx1), (float)(h.dy2 - h.dy1)));
    return h;
}

// calcHaarPattern (src/surf.cpp:128-134), n = 2: double accumulation of float products
__device__ __forceinline__ float haar2(const int32_t *S, int stride, const HaarBox &h0, const HaarBox &h1) {
    auto box = [&](const HaarBox &h) {
        const int v = S[h.dy1 * stride + h.dx1] + S[h.dy2 * stride + h.dx2] - S[h.dy2 * stride + h.dx1] - S[h.dy1 * stride + h.dx2];
        return (double)__fmul_rn((float)v, h.w);
    };
    return (float)__dadd_rn(__dadd_rn(0.0, box(h0)), box(h1));
}

struct AreaCell { int s_first, n_mid, has_first, has_last; float a_first, a_mid, a_last; };

// computeResizeAreaTab (OpenCV resize.cpp) for destination index d of a S -> 21 decimation
__device__ __forceinline__ AreaCell area_cell(int d, int S) {
    const double scale = (double)S / PW;
    const double fsx1 = d * scale, fsx2 = fsx1 + scale;
    const double cw = fmin(scale, (double)S - fsx1);
    int sx1 = (int)ceil(fsx1), sx2 = (int)floor(fsx2);
    sx2 = min(sx2, S - 1);
    sx1 = min(sx1, sx2);
    AreaCell c;
    c.has_first = (sx1 - fsx1 > 1e-3);
    c.a_first = (float)((sx1 - fsx1) / cw);
    c.s_first = sx1;                       // first full source index; the partial one is s_first - 1
    c.n_mid = sx2 - sx1;
    c.a_mid = (float)(1.0 / cw);
    c.has_last = (fsx2 - sx2 > 1e-3);
    c.a_last = (float)(fmin(fmin(fsx2 - sx2, 1.0), cw) / cw);
    return c;
}

// Shared memory per warp is one arena with overlays (a keypoint's stages run one after the other):
//   [ window MAXWIN^2 u8 ][ orientation samples (x, y, angle)  |  up-scaling row buffer  |  cell sums ][ 21 x 21 patch ]
// MAXWIN = 32 serves keypoint sizes up to 11.8 px (FAST keypoints, size 7 -> 19 x 19 window: 3.2 KB per warp, so
// occupancy is bounded by registers, not by the 7.7 KB window an ORB-sized keypoint needs); MAXWIN = 88 serves the rest.
// MAXWIN = 0 (windows up to SURF_DIRECT_MAX_WIN): the window is never staged, its pixels are produced on the fly

template <int MAXWIN>
struct SurfArena {
    static constexpr int WIN = MAXWIN > 0 ? (MAXWIN * MAXWIN + 15) / 16 * 16 : 2 * SURF_DIRECT_MAX_WIN * 4;   // direct mode: per-row start positions
    static constexpr int MID = PATCH * PATCH * 8 + 512;           // 400 gradients (tx, ty) + 128 cell sums; >= 20 * PW * 4 (up-scaling rows) and 113 * 10 (orientation)
    static constexpr int PATCHB = (PW * PW + 3 + 15) / 16 * 16;
    static constexpr int BYTES = WIN + MID + PATCHB;
};

template <bool EXTENDED, int MAXWIN>
__global__ void __launch_bounds__((MAXWIN == 0 ? 2 : MAXWIN <= 32 ? S_WARPS_SMALL : S_WARPS_LARGE) * 32)
surf_describe_kernel(const uint8_t *__restrict__ img, const int32_t *__restrict__ integ, Geom g,
                     const uint32_t *__restrict__ counts, fe_kpoint *__restrict__ kp, float *__restrict__ fdesc,
                     int upright) {
    using A = SurfArena<MAXWIN>;
    constexpr int S_WARPS = MAXWIN == 0 ? 2 : MAXWIN <= 32 ? S_WARPS_SMALL : S_WARPS_LARGE;
    __shared__ __align__(16) uint8_t s_arena[S_WARPS][A::BYTES];

    const int image = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t *arena = s_arena[warp];
    uint8_t *win = arena;
    int32_t *hb = reinterpret_cast<int32_t *>(arena + A::WIN);                 // up-scaling row buffer
    float *sx_ = reinterpret_cast<float *>(arena + A::WIN);                    // orientation samples (dead before hb is written)
    float *sy_ = sx_ + N_ORI;
    int16_t *sang_ = reinterpret_cast<int16_t *>(sy_ + N_ORI);
    uint8_t *patch = arena + A::WIN + A::MID;
    const int k = blockIdx.x * S_WARPS + warp;
    if (k >= min((int)counts[image], g.kp_cap)) return;
    const size_t o = (size_t)image * g.kp_cap + k;
    const fe_kpoint key = kp[o];
    const uint8_t *src = img + (size_t)image * g.img_stride;
    const float cx = key.x, cy = key.y;
    const SurfScale sc = surf_scale(key.size);
    const int grad_wav_size = sc.grad_wav_size, win_size = sc.win_size;
    // (warp-uniform) a keypoint that is not dropped has at least one orientation sample inside the image
    const bool drop = surf_drops(cx, cy, key.size, g.w, g.h, upright != 0, MAXWIN > 0 ? MAXWIN : SURF_DIRECT_MAX_WIN);
    if (drop) {
        if (lane == 0) { kp[o].size = -1.f; }
        return;
    }
    float dir = 270.f;

    // ---- orientation (src/surf.cpp:617-670) ---------------------------------------------------------------
    if (!upright) {
        const int stride = g.w + 1;
        const int32_t *S = integ + (size_t)image * (g.h + 1) * stride;
        const HaarBox dx0 = haar_box(0, 0, 2, 4, -1, grad_wav_size), dx1 = haar_box(2, 0, 4, 4, 1, grad_wav_size);
        const HaarBox dy0 = haar_box(0, 0, 4, 2, 1, grad_wav_size), dy1 = haar_box(0, 2, 4, 4, -1, grad_wav_size);
        const float half = __fdiv_rn((float)(grad_wav_size - 1), 2.f);
        int nangle = 0;
        for (int base = 0; base < N_ORI; base += 32) {
            const int kk = base + lane;
            bool ok = false;
            float X = 0.f, Y = 0.f;
            if (kk < N_ORI) {
                int x, y;
                ok = surf_ori_sample(cx, cy, sc, half, d_apt[kk][0], d_apt[kk][1], g.w, g.h, x, y);
                if (ok) {
                    const int32_t *ptr = S + (size_t)y * stride + x;
                    const float vx = haar2(ptr, stride, dx0, dx1), vy = haar2(ptr, stride, dy0, dy1);
                    X = __fmul_rn(vx, d_aptw[kk]);
                    Y = __fmul_rn(vy, d_aptw[kk]);
                }
            }
            const uint32_t m = __ballot_sync(0xffffffffu, ok);
            if (ok) {
                const int pos = nangle + __popc(m & ((1u << lane) - 1u));
                sx_[pos] = X;
                sy_[pos] = Y;
                sang_[pos] = (int16_t)__float2int_rn(fast_atan2_deg(Y, X));
            }
            nangle += __popc(m);
        }
        __syncwarp();
        {
            // 72 windows of 60 degrees, 5 degrees apart; lane handles windows lane, lane+32, lane+64
            float best_mod = 0.f, bestx = 0.f, besty = 0.f;
            int best_i = 1 << 30;
            for (int wi = lane; wi < 72; wi += 32) {
                const int i = wi * 5;
                float sumx = 0.f, sumy = 0.f;
                for (int j = 0; j < nangle; ++j) {
                    const int d = abs((int)sang_[j] - i);
                    if (d < 30 || d > 330) {
                        sumx = __fadd_rn(sumx, sx_[j]);
                        sumy = __fadd_rn(sumy, sy_[j]);
                    }
                }
                const float mod = __fadd_rn(__fmul_rn(sumx, sumx), __fmul_rn(sumy, sumy));
                if (mod > best_mod) { best_mod = mod; bestx = sumx; besty = sumy; best_i = i; }
            }
            // first window (smallest i) with the strictly largest modulus; all-zero keeps (0, 0)
#pragma unroll
            for (int off = 16; off; off >>= 1) {
                const float om = __shfl_xor_sync(0xffffffffu, best_mod, off);
                const float ox = __shfl_xor_sync(0xffffffffu, bestx, off);
                const float oy = __shfl_xor_sync(0xffffffffu, besty, off);
                const int oi = __shfl_xor_sync(0xffffffffu, best_i, off);
                if (om > best_mod || (om == best_mod && oi < best_i)) { best_mod = om; bestx = ox; besty = oy; best_i = oi; }
            }
            dir = fast_atan2_deg(-besty, bestx);
        }
    }
    if (lane == 0) kp[o].angle = dir;

    // ---- window extraction (src/surf.cpp:675-769) -----------------------------------------------------------
    __syncwarp();
    const float win_offset = -__fdiv_rn((float)(win_size - 1), 2.f);
    // direct mode (MAXWIN == 0, keypoints of the Fast-Hessian detector: windows of hundreds of pixels): the window is
    // not staged; win_at(i, j) below reproduces WIN[i * win_size + j] of src/surf.cpp:713-768 on the fly
    int up_start_x = 0, up_start_y = 0;
    float rot_sin = 0.f, rot_cos = 0.f;
    float *row_sx = reinterpret_cast<float *>(arena), *row_sy = row_sx + SURF_DIRECT_MAX_WIN;
    if (MAXWIN == 0) {
        if (upright) {
            up_start_x = __float2int_rn(__fadd_rn(cx, win_offset));
            up_start_y = __float2int_rn(__fsub_rn(cy, win_offset));
        } else {
            const float d = __fmul_rn(dir, (float)(3.14159265358979323846 / 180.0));
            rot_sin = -(float)sin((double)d); rot_cos = (float)cos((double)d);
            if (lane == 0) {       // start_x += sin_dir, start_y += cos_dir: sequential float additions (src/surf.cpp:724-725)
                float sxv = __fadd_rn(__fadd_rn(cx, __fmul_rn(win_offset, rot_cos)), __fmul_rn(win_offset, rot_sin));
                float syv = __fadd_rn(__fsub_rn(cy, __fmul_rn(win_offset, rot_sin)), __fmul_rn(win_offset, rot_cos));
                for (int i = 0; i < win_size; ++i) {
                    row_sx[i] = sxv; row_sy[i] = syv;
                    sxv = __fadd_rn(sxv, rot_sin); syv = __fadd_rn(syv, rot_cos);
                }
            }
        }
        __syncwarp();
    }
    auto win_at = [&](int i, int j) -> float {
        if (MAXWIN > 0) return (float)win[i * win_size + j];
        if (upright) {
            const int x = min(max(up_start_x + i, 0), g.w - 1), y = min(max(up_start_y - j, 0), g.h - 1);
            return (float)src[(size_t)y * g.pitch + x];
        }
        // pixel_x += cos_dir, pixel_y -= sin_dir in double; evaluated as start + j * step (the j sequential additions of
        // the reference differ from this by ~1e-13 px, which can only matter exactly on a pixel boundary)
        const double px = (double)row_sx[i] + (double)j * (double)rot_cos, py = (double)row_sy[i] - (double)j * (double)rot_sin;
        const int ix = (int)floor(px), iy = (int)floor(py);
        const int ncols1 = g.w - 1, nrows1 = g.h - 1;
        if ((unsigned)ix < (unsigned)ncols1 && (unsigned)iy < (unsigned)nrows1) {
            const float a = (float)(px - ix), b = (float)(py - iy);
            const uint8_t *p = src + (size_t)iy * g.pitch + ix;
            const float a1 = __fsub_rn(1.f, a), b1 = __fsub_rn(1.f, b);
            float v = __fmul_rn(__fmul_rn((float)p[0], a1), b1);
            v = __fadd_rn(v, __fmul_rn(__fmul_rn((float)p[1], a), b1));
            v = __fadd_rn(v, __fmul_rn(__fmul_rn((float)p[g.pitch], a1), b));
            v = __fadd_rn(v, __fmul_rn(__fmul_rn((float)p[g.pitch + 1], a), b));
            return (float)(uint8_t)__float2int_rn(v);
        }
        const int x = min(max((int)rint(px), 0), ncols1), y = min(max((int)rint(py), 0), nrows1);
        return (float)src[(size_t)y * g.pitch + x];
    };
    if (MAXWIN > 0) {
        if (upright) {
            const int start_x = __float2int_rn(__fadd_rn(cx, win_offset));
            const int start_y = __float2int_rn(__fsub_rn(cy, win_offset));
            // lane = window column i (image x), rows j walk up the image: every step reads win_size consecutive bytes
            if (start_x >= 0 && start_x + win_size <= g.w && start_y - (win_size - 1) >= 0 && start_y < g.h) {
                // window inside the image (warp-uniform): no clamps, a running row pointer
                for (int i = lane; i < win_size; i += 32) {
                    const uint8_t *p = src + (size_t)start_y * g.pitch + (start_x + i);
                    uint8_t *wrow = win + i * win_size;
                    for (int j = 0; j < win_size; ++j) { wrow[j] = *p; p -= g.pitch; }
                }
            } else {
                for (int i = lane; i < win_size; i += 32) {
                    const uint8_t *col = src + min(max(start_x + i, 0), g.w - 1);
                    uint8_t *wrow = win + i * win_size;
                    for (int j = 0; j < win_size; ++j) wrow[j] = col[(size_t)min(max(start_y - j, 0), g.h - 1) * g.pitch];
                }
            }
        } else {
            const float d = __fmul_rn(dir, (float)(3.14159265358979323846 / 180.0));
            const float sin_dir = -(float)sin((double)d), cos_dir = (float)cos((double)d);
            const float sx0 = __fadd_rn(__fadd_rn(cx, __fmul_rn(win_offset, cos_dir)), __fmul_rn(win_offset, sin_dir));
            const float sy0 = __fadd_rn(__fsub_rn(cy, __fmul_rn(win_offset, sin_dir)), __fmul_rn(win_offset, cos_dir));
            const int ncols1 = g.w - 1, nrows1 = g.h - 1;
            for (int i = lane; i < win_size; i += 32) {
                // start_x += sin_dir, start_y += cos_dir: i sequential float additions
                float start_x = sx0, start_y = sy0;
                for (int t = 0; t < i; ++t) { start_x = __fadd_rn(start_x, sin_dir); start_y = __fadd_rn(start_y, cos_dir); }
                double px = (double)start_x, py = (double)start_y;
                for (int j = 0; j < win_size; ++j) {
                    const int ix = (int)floor(px), iy = (int)floor(py);
                    uint8_t out;
                    if ((unsigned)ix < (unsigned)ncols1 && (unsigned)iy < (unsigned)nrows1) {
                        const float a = (float)(px - ix), b = (float)(py - iy);
                        const uint8_t *p = src + (size_t)iy * g.pitch + ix;
                        const float a1 = __fsub_rn(1.f, a), b1 = __fsub_rn(1.f, b);
                        float v = __fmul_rn(__fmul_rn((float)p[0], a1), b1);
                        v = __fadd_rn(v, __fmul_rn(__fmul_rn((float)p[1], a), b1));
                        v = __fadd_rn(v, __fmul_rn(__fmul_rn((float)p[g.pitch], a1), b));
                        v = __fadd_rn(v, __fmul_rn(__fmul_rn((float)p[g.pitch + 1], a), b));
                        out = (uint8_t)__float2int_rn(v);
                    } else {
                        const int x = min(max((int)rint(px), 0), ncols1), y = min(max((int)rint(py), 0), nrows1);
                        out = src[(size_t)y * g.pitch + x];
                    }
                    win[i * win_size + j] = out;
                    px += (double)cos_dir;
                    py -= (double)sin_dir;
                }
            }
        }
    }
    __syncwarp();

    // ---- resize(win, 21 x 21, INTER_AREA) (src/surf.cpp:772) ------------------------------------------------
    const int S = win_size;
    bool fused_grad = false;
    if (MAXWIN > 0 && S == PW) {
        for (int idx = lane; idx < PW * PW; idx += 32) patch[idx] = win[idx];
    } else if (MAXWIN > 0 && S < PW) {
        // bilinear with area-mode coefficients, INTER_RESIZE_COEF_BITS = 11; lane = destination column/row
        int sx = 0, a0 = 2048, a1 = 0;
        if (lane < PW) { const UpCoef c = d_up[S][lane]; sx = c.sx; a0 = c.a0; a1 = c.a1; }    // host-built table (upload_tables)
        // Both passes FUSED with the gradients, nothing but the window in shared memory: lane = patch column.  The rows'
        // source index sy(dy) (the same table serves rows and columns: square window) never decreases and grows by at most
        // one per step when up-scaling, so the two horizontally interpolated source rows a patch row needs ROLL through two
        // registers (hA = row sy, hB = row min(sy + 1, S - 1)); patch row dy is produced in registers, its right neighbour
        // comes by shuffle, the row above from the previous step.  Neither the row buffer nor the 21 x 21 patch is stored.
        float2 *gradf = reinterpret_cast<float2 *>(arena + A::WIN);
        const int sx1 = min(sx + 1, S - 1);
        const uint8_t *wc0 = win + sx, *wc1 = win + sx1;
        auto hrow = [&](int r) { return (int)wc0[r * S] * a0 + (int)wc1[r * S] * a1; };
        int r0 = 0, hA = hrow(0), hB = hrow(min(1, S - 1));
        int vp = 0, vpr = 0;
#pragma unroll
        for (int dy = 0; dy < PW; ++dy) {
            const int sy = __shfl_sync(0xffffffffu, sx, dy), b0 = __shfl_sync(0xffffffffu, a0, dy),
                      b1 = __shfl_sync(0xffffffffu, a1, dy);
            if (sy > r0) { r0 = sy; hA = hB; hB = hrow(min(sy + 1, S - 1)); }      // warp-uniform
            const int v = ((((b0 * (hA >> 4)) >> 16) + ((b1 * (hB >> 4)) >> 16) + 2) >> 2) & 0xFF;
            const int vr = __shfl_down_sync(0xffffffffu, v, 1);
            if (dy > 0 && lane < PATCH) {
                const int idx = (dy - 1) * PATCH + lane;
                const float dw = d_dw[idx];
                // p00 = vp, p01 = vpr, p10 = v, p11 = vr
                gradf[idx] = make_float2(__fmul_rn((float)(vpr - vp + vr - v), dw), __fmul_rn((float)(v - vp + vr - vpr), dw));
            }
            vp = v; vpr = vr;
        }
        fused_grad = true;
    } else if (S % PW == 0) {
        // integer decimation (cv::resize's is_area_fast): int box sums; x2 is ResizeAreaFastVec's (a+b+c+d+2)>>2, larger
        // factors are ResizeAreaFast_Invoker's saturate_cast<uchar>(sum * (1.f / area)), i.e. round half even.  win_size 42
        // is every keypoint of size 15 (the second Fast-Hessian filter), so this path is a common one; lane = dx
        const int kdec = S / PW;
        const float inv_area = __fdiv_rn(1.f, (float)(kdec * kdec));
        for (int dy = 0; dy < PW; ++dy) {
            int box = 0;
            if (lane < PW)
                for (int r = 0; r < kdec; ++r)
                    for (int c = 0; c < kdec; ++c) box += (int)win_at(dy * kdec + r, lane * kdec + c);
            const int v = kdec == 2 ? (box + 2) >> 2 : __float2int_rn(__fmul_rn((float)box, inv_area));
            if (lane < PW) patch[dy * PW + lane] = (uint8_t)min(max(v, 0), 255);
        }
    } else {
        // general area decimation: dst(dy, dx) = sum_j beta_j * (sum_i alpha_i * win[sy_j][sx_i]), float, in
        // table order (first partial cell, full cells, last partial cell); lane = dx
        AreaCell cx_ = area_cell(min(lane, PW - 1), S);
        for (int dy = 0; dy < PW; ++dy) {
            const AreaCell cy_ = area_cell(dy, S);
            float sum = 0.f;
            bool first_row = true;
            auto row_buf = [&](int sy) {
                float buf = 0.f;
                if (cx_.has_first) buf = __fadd_rn(buf, __fmul_rn(win_at(sy, cx_.s_first - 1), cx_.a_first));
                for (int t = 0; t < cx_.n_mid; ++t) buf = __fadd_rn(buf, __fmul_rn(win_at(sy, cx_.s_first + t), cx_.a_mid));
                if (cx_.has_last) buf = __fadd_rn(buf, __fmul_rn(win_at(sy, cx_.s_first + cx_.n_mid), cx_.a_last));
                return buf;
            };
            auto acc = [&](int sy, float beta) {
                const float t = __fmul_rn(beta, row_buf(sy));
                sum = first_row ? t : __fadd_rn(sum, t);
                first_row = false;
            };
            if (cy_.has_first) acc(cy_.s_first - 1, cy_.a_first);
            for (int t = 0; t < cy_.n_mid; ++t) acc(cy_.s_first + t, cy_.a_mid);
            if (cy_.has_last) acc(cy_.s_first + cy_.n_mid, cy_.a_last);
            if (lane < PW) patch[dy * PW + lane] = (uint8_t)min(max(__float2int_rn(sum), 0), 255);
        }
    }
    __syncwarp();

    // ---- gradients + 4 x 4 cells (src/surf.cpp:775-843) --------------------------------------------------------
    // All 32 lanes first produce the 400 weighted gradients (tx, ty); then two lanes share a cell: one owns the sums fed by
    // tx, the other those fed by ty.  Every accumulator still receives its samples in raster order, one rounding per
    // addition, exactly as the reference's loop does.
    constexpr int NB = EXTENDED ? 8 : 4;
    float2 *grad = reinterpret_cast<float2 *>(arena + A::WIN);                 // 400 x (tx, ty); hb is dead by now
    float *svec = reinterpret_cast<float *>(arena + A::WIN + PATCH * PATCH * 8);
    for (int idx = lane; idx < (fused_grad ? 0 : PATCH * PATCH); idx += 32) {
        const int y = idx / PATCH, x = idx - y * PATCH;
        const int p00 = patch[y * PW + x], p01 = patch[y * PW + x + 1], p10 = patch[(y + 1) * PW + x],
                  p11 = patch[(y + 1) * PW + x + 1];
        const float dw = d_dw[idx];
        grad[idx] = make_float2(__fmul_rn((float)(p01 - p00 + p11 - p10), dw), __fmul_rn((float)(p10 - p00 + p11 - p01), dw));
    }
    __syncwarp();
    {
        const int cell = lane >> 1, half = lane & 1;
        const int ci = cell >> 2, cj = cell & 3;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        for (int y = ci * 5; y < ci * 5 + 5; ++y)
#pragma unroll
            for (int x = 0; x < 5; ++x) {
                const float2 t = grad[y * PATCH + cj * 5 + x];
                const float u = half ? t.y : t.x, sgn = half ? t.x : t.y;
                if (EXTENDED) {
                    if (sgn >= 0) { a0 = __fadd_rn(a0, u); a1 = __fadd_rn(a1, fabsf(u)); }
                    else { a2 = __fadd_rn(a2, u); a3 = __fadd_rn(a3, fabsf(u)); }
                } else {
                    a0 = __fadd_rn(a0, u); a1 = __fadd_rn(a1, fabsf(u));
                }
            }
        if (EXTENDED) {
            float *o4 = svec + cell * 8 + half * 4;         // v[0..3] = tx sums by sign of ty, v[4..7] = ty sums by sign of tx
            o4[0] = a0; o4[1] = a1; o4[2] = a2; o4[3] = a3;
        } else {
            svec[cell * 4 + half] = a0;                      // v[0] = sum tx, v[1] = sum ty
            svec[cell * 4 + 2 + half] = a1;                  // v[2] = sum |tx|, v[3] = sum |ty|
        }
    }
    __syncwarp();
    // square_mag (src/surf.cpp:815-816,839-840) in double; summed lane-parallel + butterfly instead of sequentially
    // (a 1e-16 relative difference, far inside the 1e-4 descriptor tolerance)
    double sq = 0.0;
    for (int q = lane; q < 16 * NB; q += 32) sq = __dadd_rn(sq, (double)__fmul_rn(svec[q], svec[q]));
#pragma unroll
    for (int off = 16; off; off >>= 1) sq = __dadd_rn(sq, __shfl_xor_sync(0xffffffffu, sq, off));
    const float scale = (float)(1.0 / (sqrt(sq) + 2.220446049250313e-16));
    float *out = fdesc + o * 128;
    for (int q = lane; q < 16 * NB; q += 32) out[q] = __fmul_rn(svec[q], scale);
}

int launch_integral(const Geom &g, const Buffers &b, cudaStream_t s) {
    dim3 rgrid(div_up(g.h, 8), g.n_images);
    integral_rows_kernel<<<rgrid, 256, 0, s>>>(b.img, b.integral, g);
    dim3 cgrid(div_up(g.w + 1, 128), g.n_images);
    integral_cols_kernel<<<cgrid, 128, 0, s>>>(b.integral, g);
    return 2;
}

int launch_surf(const Geom &g, const Buffers &b, const uint32_t *counts, bool extended, bool upright, int max_win,
                cudaStream_t s) {
    upload_tables();
    int n = 0;
    if (!upright) {
        dim3 rgrid(div_up(g.h, 8), g.n_images);
        integral_rows_kernel<<<rgrid, 256, 0, s>>>(b.img, b.integral, g);
        dim3 cgrid(div_up(g.w + 1, 128), g.n_images);
        integral_cols_kernel<<<cgrid, 128, 0, s>>>(b.integral, g);
        n += 2;
    }
    const int warps = max_win <= 32 ? S_WARPS_SMALL : max_win <= SURF_MAX_WIN ? S_WARPS_LARGE : 2;
    dim3 grid(div_up(g.kp_cap, warps), g.n_images);
    const int up = upright ? 1 : 0;
#define FE_SURF_GO(EXT, MW) surf_describe_kernel<EXT, MW><<<grid, warps * 32, 0, s>>>(b.img, b.integral, g, counts, b.kp, b.fdesc, up)
    if (max_win <= 32) { if (extended) FE_SURF_GO(true, 32); else FE_SURF_GO(false, 32); }
    else if (max_win <= SURF_MAX_WIN) { if (extended) FE_SURF_GO(true, SURF_MAX_WIN); else FE_SURF_GO(false, SURF_MAX_WIN); }
    else { if (extended) FE_SURF_GO(true, 0); else FE_SURF_GO(false, 0); }
#undef FE_SURF_GO
    return n + 1;
}

}  // namespace fe
