// BRIEF-16 / 32 / 64 descriptors (cv::BriefDescriptorExtractor) with a caller-supplied test pattern.
//
// Replaces  cv::BriefDescriptorExtractor extractor(16); extractor.compute(img, kps, desc)  of the reference's live C++
// node (/root/reference src/live_stereo.cpp:238,359-360) and  cv2.xfeatures2d.BriefDescriptorExtractor_create(bytes,
// use_orientation)  of the Python descriptor table (src/front_end/features.py:93-96, bin/detect_node:28-29).
//
// Algorithm (OpenCV features2d/src/brief.cpp, 2.4 and contrib): PATCH_SIZE 48, KERNEL_SIZE 9; keypoints closer than
// 48/2 + 9/2 = 28 px to the border are removed; integral image CV_32S; test i compares two 9 x 9 box sums
//     smoothedSum(y, x) = S(Y+5, X+5) - S(Y+5, X-4) - S(Y-4, X+5) + S(Y-4, X-4),  Y = (int)(pt.y + 0.5) + y, X likewise,
// bit (7 - i % 8) of byte i / 8 is  smoothedSum(y1, x1) < smoothedSum(y2, x2)  (the first test of a byte is its MSB).
// The (y1, x1, y2, x2) tables (generated_16.i / _32.i / _64.i) live in OpenCV's sources, which are not in this image:
// the caller supplies them (fe_set_brief_pattern) -- PARITY UNPINNED for the table, the arithmetic is integer-exact.
// use_orientation (contrib only): the offsets are rotated by kp.angle and clamped to +-24 before use.
//
// One warp per keypoint: lane l evaluates tests l, l + 32, ...; a ballot is 32 tests = 4 descriptor bytes after a
// bit reversal inside every byte.  The pattern sits in shared memory; the eight corner reads per test go to the L1/L2-
// resident integral image (the 57 x 57 window of a keypoint is 13 KB of it).
#include "fe_internal.cuh"

namespace fe {

constexpr int BF_WARPS = 8, BF_KPW = 4;      // warps per CTA, keypoints per warp

__global__ void __launch_bounds__(BF_WARPS * 32)
brief_kernel(const int32_t *__restrict__ integ, Geom g, const uint32_t *__restrict__ counts, const fe_kpoint *__restrict__ kp,
             const int8_t *__restrict__ pattern, int bytes, int use_orientation, uint8_t *__restrict__ out) {
    __shared__ int8_t s_pat[512 * 4];
    const int n_tests = bytes * 8;
    for (int i = threadIdx.x; i < n_tests; i += blockDim.x)
        reinterpret_cast<uint32_t *>(s_pat)[i] = reinterpret_cast<const uint32_t *>(pattern)[i];
    __syncthreads();
    const int image = blockIdx.y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = min((int)counts[image], g.kp_cap);
    const int stride = g.w + 1;
    const int32_t *S = integ + (size_t)image * (g.h + 1) * stride;
    for (int kk = 0; kk < BF_KPW; ++kk) {
        const int k = (blockIdx.x * BF_WARPS + warp) * BF_KPW + kk;
        if (k >= n) return;
        const fe_kpoint key = kp[(size_t)image * g.kp_cap + k];
        const int cy = (int)((double)key.y + 0.5), cx = (int)((double)key.x + 0.5);
        float r0 = 0.f, r1 = 1.f;
        if (use_orientation) {
            const float2 cs = steer(key.angle);
            r0 = cs.y;
            r1 = cs.x;
        }
        uint32_t *dst = reinterpret_cast<uint32_t *>(out + ((size_t)image * g.kp_cap + k) * 64);
        for (int base = 0; base < n_tests; base += 32) {
            const char4 t = reinterpret_cast<const char4 *>(s_pat)[base + lane];       // (y1, x1, y2, x2)
            int y1 = t.x, x1 = t.y, y2 = t.z, x2 = t.w;
            if (use_orientation) {
                auto rot = [&](int &y, int &x) {
                    const int rx = (int)__fsub_rn(__fmul_rn((float)x, r1), __fmul_rn((float)y, r0));
                    const int ry = (int)__fadd_rn(__fmul_rn((float)x, r0), __fmul_rn((float)y, r1));
                    x = min(max(rx, -24), 24);
                    y = min(max(ry, -24), 24);
                };
                rot(y1, x1);
                rot(y2, x2);
            }
            auto smoothed = [&](int y, int x) {
                // rows Y - 4 and min(Y + 5, h), columns X - 4 and min(X + 5, w): a coordinate that rounds up onto the 28-px
                // border with an offset of +24 would index one past the integral image (OpenCV reads out of bounds there)
                const int ya = cy + y - 4, xa = cx + x - 4, yb = min(ya + 9, g.h), xb = min(xa + 9, g.w);
                const int32_t *pa = S + (size_t)ya * stride, *pb = S + (size_t)yb * stride;
                return __ldg(pb + xb) - __ldg(pb + xa) - __ldg(pa + xb) + __ldg(pa + xa);
            };
            const uint32_t bal = __ballot_sync(0xffffffffu, smoothed(y1, x1) < smoothed(y2, x2));
            // test 32 m + 8 b + j -> byte 4 m + b, bit 7 - j: reverse the bits inside every byte of the ballot
            if (lane == 0) dst[base >> 5] = __byte_perm(__brev(bal), 0, 0x0123);
        }
    }
}

int launch_brief_ext(const Geom &g, const Buffers &b, const uint32_t *counts, const int8_t *pattern, int bytes, int use_orientation,
                     uint8_t *out, cudaStream_t s) {
    dim3 grid(div_up(g.kp_cap, BF_WARPS * BF_KPW), g.n_images);
    brief_kernel<<<grid, BF_WARPS * 32, 0, s>>>(b.integral, g, counts, b.kp, pattern, bytes, use_orientation, out);
    return 1;
}

}  // namespace fe
