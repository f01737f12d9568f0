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
// Two kernels compute the same bits.  Both evaluate 32 tests per warp round: lane l takes test l of the round, and a ballot is
// 4 descriptor bytes after a bit reversal inside every byte.  The pattern sits in shared memory.
//   brief_kernel       one warp per keypoint, any keypoint order; eight corner reads per test from the L1/L2-resident integral
//                      image (the 57 x 57 window of a keypoint is 13 KB of it).  fe_describe, and the batch under a pyramid.
//   brief_tile_kernel  one CTA per image tile of raster-ordered keypoints; the tile's 9 x 9 box sums are formed once in shared
//                      memory, so a test is two shared-memory reads.  The single-level batch and fe_stereo_features.
// The batch applies the 28-px border on the device (brief_border_kernel) after detection, as compute() does after detect().
#include "fe_internal.cuh"

namespace fe {

constexpr int BF_WARPS = 8, BF_KPW = 4;      // warps per CTA, keypoints per warp
constexpr int BRIEF_BORDER = 48 / 2 + 9 / 2;  // PATCH_SIZE / 2 + KERNEL_SIZE / 2 = 28
constexpr int BRIEF_REACH = 24;               // largest |test offset|: tables are checked, rotated offsets clamped

// KeyPointsFilter::runByImageBorder(keypoints, image.size(), 28) on the float coordinates
__device__ __forceinline__ bool brief_keeps(float x, float y, int w, int h) {
    return x >= BRIEF_BORDER && x < w - BRIEF_BORDER && y >= BRIEF_BORDER && y < h - BRIEF_BORDER;
}

// The keypoint's rotation (sin, cos) of its angle in degrees, and the rotated test: contrib's use_orientation rotates both
// points by kp.angle, truncates them to int and clamps them to +-24.  Without orientation the test is used as is.
__device__ __forceinline__ int4 brief_test(char4 t, bool orient, float2 rot) {
    int4 r = make_int4(t.x, t.y, t.z, t.w);               // (y1, x1, y2, x2)
    if (orient) {
        auto turn = [&](int &y, int &x) {
            const int rx = (int)__fsub_rn(__fmul_rn((float)x, rot.y), __fmul_rn((float)y, rot.x));
            const int ry = (int)__fadd_rn(__fmul_rn((float)x, rot.x), __fmul_rn((float)y, rot.y));
            x = min(max(rx, -BRIEF_REACH), BRIEF_REACH);
            y = min(max(ry, -BRIEF_REACH), BRIEF_REACH);
        };
        turn(r.x, r.y);
        turn(r.z, r.w);
    }
    return r;
}
__device__ __forceinline__ float2 brief_rotation(float angle_deg) {
    const float2 cs = steer(angle_deg);
    return make_float2(cs.y, cs.x);
}
// test 32 m + 8 b + j -> byte 4 m + b, bit 7 - j: reverse the bits inside every byte of the ballot
__device__ __forceinline__ uint32_t brief_word(uint32_t ballot) { return __byte_perm(__brev(ballot), 0, 0x0123); }

__global__ void __launch_bounds__(BF_WARPS * 32)
brief_kernel(const int32_t *__restrict__ integ, Geom g, const uint32_t *__restrict__ counts, const fe_kpoint *__restrict__ kp,
             const int8_t *__restrict__ pattern, int bytes, int use_orientation, uint8_t *__restrict__ out, int row_bytes) {
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
        const float2 rot = use_orientation ? brief_rotation(key.angle) : make_float2(0.f, 1.f);
        uint32_t *dst = reinterpret_cast<uint32_t *>(out + ((size_t)image * g.kp_cap + k) * row_bytes);
        for (int base = 0; base < n_tests; base += 32) {
            const int4 t = brief_test(reinterpret_cast<const char4 *>(s_pat)[base + lane], use_orientation, rot);
            auto smoothed = [&](int y, int x) {
                // rows Y - 4 and min(Y + 5, h), columns X - 4 and min(X + 5, w): a coordinate that rounds up onto the 28-px
                // border with an offset of +24 would index one past the integral image (OpenCV reads out of bounds there)
                const int ya = cy + y - 4, xa = cx + x - 4, yb = min(ya + 9, g.h), xb = min(xa + 9, g.w);
                const int32_t *pa = S + (size_t)ya * stride, *pb = S + (size_t)yb * stride;
                return __ldg(pb + xb) - __ldg(pb + xa) - __ldg(pa + xb) + __ldg(pa + xa);
            };
            const uint32_t bal = __ballot_sync(0xffffffffu, smoothed(t.x, t.y) < smoothed(t.z, t.w));
            if (lane == 0) dst[base >> 5] = brief_word(bal);
        }
        if (lane < (row_bytes - bytes) / 4) dst[bytes / 4 + lane] = 0u;      // zero padding of narrower rows
    }
}

int launch_brief_ext(const Geom &g, const Buffers &b, const uint32_t *counts, const int8_t *pattern, int bytes, int use_orientation,
                     uint8_t *out, int row_bytes, cudaStream_t s) {
    dim3 grid(div_up(g.kp_cap, BF_WARPS * BF_KPW), g.n_images);
    brief_kernel<<<grid, BF_WARPS * 32, 0, s>>>(b.integral, g, counts, b.kp, pattern, bytes, use_orientation, out, row_bytes);
    return 1;
}

// ---- the batch: 28-px border on the device ------------------------------------------------------------------------------
// One CTA per image: the keypoints that BriefDescriptorExtractor::compute keeps, compacted in place and in order (ballots and
// one block scan per 1024 entries; a chunk is read whole before any of its entries is written, and it is written only at or
// before its own positions).  Runs after the detector's top-N / Harris cut, so it removes keypoints from the list the
// detector returned.  What later stages read moves with the keypoint: the record, its raster key, kx / ky.  An image whose
// count exceeds kp_cap is left as it is: the count reports the overflow.
constexpr int BB_THREADS = 1024;

__global__ void __launch_bounds__(BB_THREADS)
brief_border_kernel(Geom g, uint32_t *__restrict__ n_kp, fe_kpoint *__restrict__ kp, uint32_t *__restrict__ kp_key,
                    float *__restrict__ kx, float *__restrict__ ky) {
    __shared__ uint32_t s_warp[33];
    const int image = blockIdx.x;
    const uint32_t count = n_kp[image];
    if (count > (uint32_t)g.kp_cap) return;
    const int n = (int)count;
    const size_t o = (size_t)image * g.kp_cap;
    uint32_t kept = 0;
    for (int base = 0; base < n; base += BB_THREADS) {
        const int i = base + threadIdx.x;
        fe_kpoint k{};
        uint32_t key = 0;
        float x = 0.f, y = 0.f;
        bool keep = false;
        if (i < n) {
            k = kp[o + i]; key = kp_key[o + i]; x = kx[o + i]; y = ky[o + i];
            keep = brief_keeps(k.x, k.y, g.w, g.h);
        }
        uint32_t total;
        const uint32_t pos = kept + block_excl_scan_1024(keep ? 1u : 0u, s_warp, total);    // (its barriers: every read is done)
        if (keep) { kp[o + pos] = k; kp_key[o + pos] = key; kx[o + pos] = x; ky[o + pos] = y; }
        kept += total;
    }
    if (threadIdx.x == 0) n_kp[image] = kept;
}

int launch_brief_border(const Geom &g, const Buffers &b, cudaStream_t s) {
    brief_border_kernel<<<g.n_images, BB_THREADS, 0, s>>>(g, b.n_kp, b.kp, b.kp_key, b.kx, b.ky);
    return 1;
}

// ---- BRIEF per image tile -----------------------------------------------------------------------------------------------
// One CTA per (image, BT_ROWS x BT_COLS tile of keypoint centres), the tile shape of orb_describe_tile_kernel.  It stages the
// raw tile with a 28-px halo (16-byte loads; pixels outside the image are 0), forms the 9 x 9 box sum of every centre the
// tests can reach (rows -24 .. +87, columns -24 .. +279 around the tile) as u16 in shared memory, and then evaluates every
// test as two shared-memory reads.  A kept keypoint has (int)(y + 0.5) <= h - 28 and offsets lie in [-24, 24], so a box runs
// past the bottom or right edge by at most one row / column, where brief_kernel clamps its integral-image index: the zeros
// give the same sums.  The sums are integers <= 81 * 255, exact in any order: the rows are bit-identical to brief_kernel's.
// Keypoints of a single-level batch sit on integer pixels (key = y << 16 | x), so (int)(kp.y + 0.5) is the key's y.
constexpr int BT_ROWS = 64, BT_COLS = 256;
constexpr int BT_HALO = BRIEF_REACH + 4;                        // 28: test offset + half box
constexpr int BT_XL = 32;                                       // raw columns start at x0 - 32 (16-byte aligned, >= 28)
constexpr int BT_RAW_ROWS = BT_ROWS + 2 * BT_HALO;             // 120: rows y0 - 28 .. y0 + 91
constexpr int BT_RAW_B = BT_COLS + 2 * BT_XL;                  // 320 bytes per raw row: x0 - 32 .. x0 + 287
constexpr int BT_VECS = BT_RAW_B / 16;
constexpr int BT_BOX_ROWS = BT_ROWS + 2 * BRIEF_REACH;         // 112 box centres: y0 - 24 .. y0 + 87
constexpr int BT_BOX_COLS = BT_COLS + 2 * BRIEF_REACH;         // 304 box centres: x0 - 24 .. x0 + 279
constexpr int BT_WARPS = 10, BT_THREADS = BT_WARPS * 32;       // one thread per box column
constexpr int BT_CHUNK = 2 * BT_THREADS;                        // entries of the tile's row band examined per pass
constexpr int BT_STAGE = (BT_RAW_ROWS * BT_VECS + BT_THREADS - 1) / BT_THREADS;   // 16-byte loads per thread
constexpr int BT_RAW_SMEM = BT_RAW_ROWS * BT_RAW_B;            // 38 400 B
constexpr int BT_SMEM = BT_RAW_SMEM + BT_BOX_ROWS * BT_BOX_COLS * 2;    // + 68 096 B of box sums: dynamic
static_assert(BT_BOX_COLS <= BT_THREADS, "one thread per box column");
static_assert(BT_COLS % 16 == 0 && BT_XL % 16 == 0 && BT_XL >= BT_HALO && BT_RAW_B >= BT_XL + BT_COLS + BT_HALO, "staged columns");
static_assert(2 * BT_CHUNK * 4 <= BT_RAW_SMEM, "the keypoint list reuses the raw tile");

__global__ void __launch_bounds__(BT_THREADS, 2)
brief_tile_kernel(const uint8_t *__restrict__ img, Geom g, const uint32_t *__restrict__ n_kp, const uint32_t *__restrict__ kp_key,
                  const fe_kpoint *__restrict__ kp, const int8_t *__restrict__ pattern, int bytes, int use_orientation,
                  uint8_t *__restrict__ out, int row_bytes) {
    extern __shared__ __align__(16) uint8_t s_raw[];                                          // [BT_RAW_ROWS][BT_RAW_B]
    uint16_t *s_box = reinterpret_cast<uint16_t *>(s_raw + BT_RAW_SMEM);                    // [BT_BOX_ROWS][BT_BOX_COLS]
    __shared__ char4 s_pat[512];
    __shared__ int s_range[2], s_cnt;
    const uint32_t FULL = 0xffffffffu;
    const int image = blockIdx.z;
    const int x0 = blockIdx.x * BT_COLS, y0 = blockIdx.y * BT_ROWS;
    const int ty0 = y0 - BT_HALO, sx = x0 - BT_XL;                 // image coordinates of raw row 0 / raw byte 0
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // the raw tile, loads issued first (their latency overlaps the keypoint search)
    uint4 v[BT_STAGE];
#pragma unroll
    for (int k = 0; k < BT_STAGE; ++k) {
        const int i = threadIdx.x + k * BT_THREADS, r = i / BT_VECS, c = sx + 16 * (i - r * BT_VECS), gy = ty0 + r;
        v[k] = make_uint4(0u, 0u, 0u, 0u);
        if (i < BT_RAW_ROWS * BT_VECS && gy >= 0 && gy < g.h && c >= 0 && c < g.w) {
            v[k] = __ldg(reinterpret_cast<const uint4 *>(img + (size_t)image * g.img_stride + (size_t)gy * g.pitch + c));
            if (c + 16 > g.w) {                                         // the row pitch's padding is not image: zeros
                uint32_t *wd = reinterpret_cast<uint32_t *>(&v[k]);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int valid = min(max(g.w - c - 4 * j, 0), 4);
                    wd[j] &= valid == 4 ? 0xffffffffu : (1u << (8 * valid)) - 1u;
                }
            }
        }
    }
    const int n = min((int)n_kp[image], g.kp_cap);
    const uint32_t *keys = kp_key + (size_t)image * g.kp_cap;
    if (warp < 2) {                                                 // the keypoints of rows y0 .. y0 + BT_ROWS - 1
        const int r = warp_lower_bound(keys, n, (uint32_t)(y0 + warp * BT_ROWS) << 16, lane);
        if (lane == 0) s_range[warp] = r;
    }
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    const int lo = s_range[0], hi = s_range[1];
    if (lo >= hi) return;
#pragma unroll
    for (int k = 0; k < BT_STAGE; ++k) {
        const int i = threadIdx.x + k * BT_THREADS;
        if (i < BT_RAW_ROWS * BT_VECS) *reinterpret_cast<uint4 *>(s_raw + 16 * i) = v[k];
    }
    for (int i = threadIdx.x; i < bytes * 8; i += BT_THREADS) s_pat[i] = reinterpret_cast<const char4 *>(pattern)[i];
    __syncthreads();
    // box sums, one column per thread: 9-wide row sums (three masked byte dot products) rolled 9 rows tall
    if (threadIdx.x < BT_BOX_COLS) {
        const int u = threadIdx.x, o = u & 3;
        const uint32_t *col = reinterpret_cast<const uint32_t *>(s_raw) + (u >> 2) + 1;      // raw byte u + 4 = column x0 - 28 + u
        const uint32_t m0 = 0x01010101u << (8 * o), m2 = 0x01010101u >> (8 * (3 - o));
        auto rowsum = [&](int r) {
            const uint32_t *p = col + r * (BT_RAW_B / 4);
            return __dp4a(p[0], m0, __dp4a(p[1], 0x01010101u, __dp4a(p[2], m2, 0u)));
        };
        uint32_t ring[9], acc = 0;
#pragma unroll
        for (int j = 0; j < 9; ++j) { ring[j] = rowsum(j); acc += ring[j]; }
        s_box[u] = (uint16_t)acc;
#pragma unroll 1
        for (int r0 = 9; r0 < BT_RAW_ROWS; r0 += 9) {
#pragma unroll
            for (int j = 0; j < 9; ++j) {
                const int r = r0 + j;
                if (r < BT_RAW_ROWS) {
                    const uint32_t s = rowsum(r);
                    acc += s - ring[j];
                    ring[j] = s;
                    s_box[(r - 8) * BT_BOX_COLS + u] = (uint16_t)acc;       // rows r - 8 .. r: centre row r - 4 of the raw tile
                }
            }
        }
    }
    __syncthreads();
    // the raw tile is dead: it holds the list of the tile's keypoints from here on
    uint32_t *s_idx = reinterpret_cast<uint32_t *>(s_raw), *s_key = s_idx + BT_CHUNK;
    // box sum at image (y, x): the box tile's origin is (y0 - 24, x0 - 24)
    const uint16_t *box_o = s_box - (y0 - BRIEF_REACH) * BT_BOX_COLS - (x0 - BRIEF_REACH);
    const int words = bytes / 4;
    for (int base = lo; base < hi; base += BT_CHUNK) {
        tile_collect<BT_THREADS, BT_CHUNK>(keys, base, hi, x0, BT_COLS, s_idx, s_key, &s_cnt, lane);
        __syncthreads();
        const int m = s_cnt;
        __syncthreads();
        if (threadIdx.x == 0) s_cnt = 0;
        for (int e = warp; e < m; e += BT_WARPS) {
            const uint32_t key = s_key[e];
            const size_t row = (size_t)image * g.kp_cap + s_idx[e];
            const int cy = (int)(key >> 16), cx = (int)(key & 0xFFFF);
            const float2 rot = use_orientation ? brief_rotation(kp[row].angle) : make_float2(0.f, 1.f);
            const uint16_t *centre = box_o + cy * BT_BOX_COLS + cx;
            uint32_t mine = 0;
            for (int w = 0; w < words; ++w) {
                const int4 t = brief_test(s_pat[32 * w + lane], use_orientation, rot);
                const uint32_t bal = __ballot_sync(FULL, centre[t.x * BT_BOX_COLS + t.y] < centre[t.z * BT_BOX_COLS + t.w]);
                if (lane == w) mine = brief_word(bal);
            }
            if (lane < row_bytes / 4) reinterpret_cast<uint32_t *>(out + row * row_bytes)[lane] = mine;   // (0 past `bytes`)
        }
        __syncthreads();                                            // the list is rewritten by the next pass
    }
}

int launch_brief_tile(const Geom &g, const Buffers &b, const int8_t *pattern, int bytes, int use_orientation, uint8_t *out,
                      int row_bytes, cudaStream_t s) {
    static bool smem_set[64] = {false};         // per device: the attribute belongs to the device's context
    int dev = 0;
    cudaGetDevice(&dev);
    if (!smem_set[dev & 63]) {
        cudaFuncSetAttribute(brief_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BT_SMEM);
        smem_set[dev & 63] = true;
    }
    dim3 grid(div_up(g.w, BT_COLS), div_up(g.h, BT_ROWS), g.n_images);
    brief_tile_kernel<<<grid, BT_THREADS, BT_SMEM, s>>>(b.img, g, b.n_kp, b.kp_key, b.kp, pattern, bytes, use_orientation, out,
                                                        row_bytes);
    return 1;
}

}  // namespace fe
