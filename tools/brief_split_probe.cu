// Where does rbrief_kernel's time go: staging the 39 x 39 patch from global memory, or the 512 rotated shared-memory samples?
// Times a copy of rbrief_kernel (orb.cu) three ways on the same keypoints:
//   mode 0  as it is;
//   mode 1  staging only (the patch is staged for every keypoint, no sampling);
//   mode 2  sampling only (the patch is staged once per warp, for its first keypoint, then every keypoint samples it).
// Input: a file written by tools/brief_split_probe.py (a real batch's images and its detected keypoints).  The image bytes
// stand in for the blurred image: which addresses are read does not depend on what the pixels hold.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -fmad=false -o tools/brief_split_probe tools/brief_split_probe.cu
//   ./tools/brief_split_probe batch.bin
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <cuda_runtime.h>

__device__ int8_t d_pattern[256][4] = {
#include "../front_end_b200/csrc/orb_pattern.inc"
};

constexpr int BR_WARPS = 8, BR_KPW = 8, BR_R = 19, BR_ROWS = 2 * BR_R + 1, BR_WORDS = 11, BR_STRIDE = 12;

template <int MODE>
__global__ void __launch_bounds__(BR_WARPS * 32)
brief_probe(const uint8_t *__restrict__ blur, int pitch, size_t img_stride, int kp_cap, const uint32_t *__restrict__ counts,
            const float *__restrict__ kx, const float *__restrict__ ky, const float2 *__restrict__ kcs, uint8_t *__restrict__ desc) {
    __shared__ uint32_t s_patch[BR_WARPS][BR_ROWS * BR_STRIDE];
    const int image = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = min((int)counts[image], kp_cap);
    if (blockIdx.x * (BR_WARPS * BR_KPW) >= n) return;
    float4 pat[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const char4 pt = reinterpret_cast<const char4 *>(d_pattern)[j * 32 + lane];
        pat[j] = make_float4((float)pt.x, (float)pt.y, (float)pt.z, (float)pt.w);
    }
    uint32_t *patch = s_patch[warp];
    float pre_x = 0.f, pre_y = 0.f;
    float2 pre_cs = make_float2(1.f, 0.f);
    {
        const int i = (blockIdx.x * BR_KPW + lane) * BR_WARPS + warp;
        if (lane < BR_KPW && i < n) {
            const size_t o = (size_t)image * kp_cap + i;
            pre_x = kx[o]; pre_y = ky[o]; pre_cs = kcs[o];
        }
    }
    const int st_w = lane % BR_WORDS, st_r = lane / BR_WORDS;
    const int st_goff = st_r * pitch + 4 * st_w, st_soff = st_r * BR_STRIDE + st_w;
    const int st_xoff = (3 * lane + 2) * pitch + 4 * (BR_WORDS - 1), st_xs = (3 * lane + 2) * BR_STRIDE + BR_WORDS - 1;
    constexpr uint32_t BIAS49 = 0x4B400000u * 49u;
#pragma unroll 1
    for (int it = 0; it < BR_KPW; ++it) {
        const int i = (blockIdx.x * BR_KPW + it) * BR_WARPS + warp;
        if (i >= n) break;
        const size_t o = (size_t)image * kp_cap + i;
        const int cx = __float2int_rn(__shfl_sync(0xffffffffu, pre_x, it)), cy = __float2int_rn(__shfl_sync(0xffffffffu, pre_y, it));
        const float a = __shfl_sync(0xffffffffu, pre_cs.x, it), b = __shfl_sync(0xffffffffu, pre_cs.y, it);
        const int xl = cx - BR_R, xa = xl & ~3, off = xl - xa;
        const uint8_t *base = blur + (size_t)image * img_stride + (size_t)(cy - BR_R) * pitch + xa;
        __syncwarp();
        if (MODE != 2 || it == 0) {
            const uint8_t *gp = base + st_goff;
            uint32_t *sp = patch + st_soff;
#pragma unroll
            for (int r0 = 0; r0 < BR_ROWS; r0 += 3) {
                *sp = __ldg(reinterpret_cast<const uint32_t *>(gp));
                gp += 3 * pitch; sp += 3 * BR_STRIDE;
            }
            if (lane < BR_ROWS / 3) patch[st_xs] = __ldg(reinterpret_cast<const uint32_t *>(base + st_xoff));
        }
        __syncwarp();
        if (MODE == 1) {                     // keep the staging observable: one word of the patch per lane
            if (lane < 8) reinterpret_cast<uint32_t *>(desc + o * 32)[lane] = patch[lane * 37 % (BR_ROWS * BR_STRIDE)];
            continue;
        }
        const uint8_t *pc = reinterpret_cast<const uint8_t *>(patch) + BR_R * (BR_STRIDE * 4) + BR_R + off;
        const uint32_t pcs = (uint32_t)__cvta_generic_to_shared(pc) - BIAS49;
        auto sample = [&](float fx, float fy) {
            const uint32_t bx = __float_as_uint(__fadd_rn(fx, 12582912.f)), by = __float_as_uint(__fadd_rn(fy, 12582912.f));
            uint32_t v;
            asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(pcs + by * (uint32_t)(BR_STRIDE * 4) + bx));
            return v;
        };
        uint32_t word = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float4 pt = pat[j];
            const float x0 = pt.x, y0 = pt.y, x1 = pt.z, y1 = pt.w;
            const uint32_t t0 = sample(__fsub_rn(__fmul_rn(x0, a), __fmul_rn(y0, b)), __fadd_rn(__fmul_rn(x0, b), __fmul_rn(y0, a)));
            const uint32_t t1 = sample(__fsub_rn(__fmul_rn(x1, a), __fmul_rn(y1, b)), __fadd_rn(__fmul_rn(x1, b), __fmul_rn(y1, a)));
            const uint32_t w = __ballot_sync(0xffffffffu, t0 < t1);
            if (lane == j) word = w;
        }
        if (lane < 8) reinterpret_cast<uint32_t *>(desc + o * 32)[lane] = word;
    }
}

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "%s: %s\n", #x, cudaGetErrorString(e_)); return 1; } } while (0)

template <int MODE>
int time_mode(const char *name, int reps, dim3 grid, const uint8_t *img, int pitch, size_t stride, int cap, const uint32_t *cnt,
              const float *kx, const float *ky, const float2 *kcs, uint8_t *desc, double base_ms) {
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
    for (int w = 0; w < 5; ++w) brief_probe<MODE><<<grid, BR_WARPS * 32>>>(img, pitch, stride, cap, cnt, kx, ky, kcs, desc);
    CK(cudaDeviceSynchronize());
    std::vector<float> t(reps);
    for (int r = 0; r < reps; ++r) {
        CK(cudaEventRecord(a));
        brief_probe<MODE><<<grid, BR_WARPS * 32>>>(img, pitch, stride, cap, cnt, kx, ky, kcs, desc);
        CK(cudaEventRecord(b));
        CK(cudaEventSynchronize(b));
        CK(cudaEventElapsedTime(&t[r], a, b));
    }
    std::sort(t.begin(), t.end());
    const double med = t[reps / 2];
    printf("%-34s median %.4f ms  min %.4f  max %.4f  (%5.1f %% of mode 0)\n", name, med, t[0], t[reps - 1],
           base_ms > 0 ? 100.0 * med / base_ms : 100.0);
    return 0;
}

int main(int argc, char **argv) {
    if (argc < 2) { fprintf(stderr, "usage: %s batch.bin\n", argv[0]); return 2; }
    FILE *f = fopen(argv[1], "rb");
    if (!f) { perror(argv[1]); return 2; }
    int32_t hdr[4];                          // n_images, w, h, kp_cap
    if (fread(hdr, 4, 4, f) != 4) return 2;
    const int NI = hdr[0], W = hdr[1], H = hdr[2], cap = hdr[3];
    const size_t img_bytes = (size_t)NI * W * H, nk = (size_t)NI * cap;
    std::vector<uint8_t> img(img_bytes);
    std::vector<uint32_t> cnt(NI);
    std::vector<float> kx(nk), ky(nk);
    std::vector<float2> kcs(nk);
    if (fread(img.data(), 1, img_bytes, f) != img_bytes || fread(cnt.data(), 4, NI, f) != (size_t)NI ||
        fread(kx.data(), 4, nk, f) != nk || fread(ky.data(), 4, nk, f) != nk || fread(kcs.data(), 8, nk, f) != nk) {
        fprintf(stderr, "short read\n");
        return 2;
    }
    fclose(f);
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, 0));
    size_t kp_total = 0;
    for (int i = 0; i < NI; ++i) kp_total += std::min<uint32_t>(cnt[i], cap);
    printf("device %s, %d SMs; %d images of %d x %d, %zu keypoints (%.0f per image)\n", prop.name, prop.multiProcessorCount, NI, W, H,
           kp_total, (double)kp_total / NI);
    uint8_t *d_img, *d_desc; uint32_t *d_cnt; float *d_kx, *d_ky; float2 *d_kcs;
    CK(cudaMalloc(&d_img, img_bytes)); CK(cudaMalloc(&d_desc, nk * 32)); CK(cudaMalloc(&d_cnt, 4 * NI));
    CK(cudaMalloc(&d_kx, 4 * nk)); CK(cudaMalloc(&d_ky, 4 * nk)); CK(cudaMalloc(&d_kcs, 8 * nk));
    CK(cudaMemcpy(d_img, img.data(), img_bytes, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_cnt, cnt.data(), 4 * NI, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_kx, kx.data(), 4 * nk, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_ky, ky.data(), 4 * nk, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_kcs, kcs.data(), 8 * nk, cudaMemcpyHostToDevice));
    const dim3 grid((cap + BR_WARPS * BR_KPW - 1) / (BR_WARPS * BR_KPW), NI);
    const size_t stride = (size_t)W * H;      // W is a multiple of 16 at the probed sizes: pitch = W
    const int reps = 200;
    // mode 0 first to get the reference time, then all three again interleaved
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
    for (int w = 0; w < 5; ++w) brief_probe<0><<<grid, BR_WARPS * 32>>>(d_img, W, stride, cap, d_cnt, d_kx, d_ky, d_kcs, d_desc);
    std::vector<float> t(reps);
    for (int r = 0; r < reps; ++r) {
        CK(cudaEventRecord(a));
        brief_probe<0><<<grid, BR_WARPS * 32>>>(d_img, W, stride, cap, d_cnt, d_kx, d_ky, d_kcs, d_desc);
        CK(cudaEventRecord(b)); CK(cudaEventSynchronize(b)); CK(cudaEventElapsedTime(&t[r], a, b));
    }
    std::sort(t.begin(), t.end());
    const double base = t[reps / 2];
    for (int round = 0; round < 2; ++round) {
        printf("round %d (%d launches per mode)\n", round, reps);
        if (time_mode<0>("0 as is", reps, grid, d_img, W, stride, cap, d_cnt, d_kx, d_ky, d_kcs, d_desc, base)) return 1;
        if (time_mode<1>("1 staging only", reps, grid, d_img, W, stride, cap, d_cnt, d_kx, d_ky, d_kcs, d_desc, base)) return 1;
        if (time_mode<2>("2 sampling only (stage once/warp)", reps, grid, d_img, W, stride, cap, d_cnt, d_kx, d_ky, d_kcs, d_desc, base)) return 1;
    }
    CK(cudaGetLastError());
    return 0;
}
