/*
 * fe_abi.h -- C-ABI of the B200-native stereo feature front-end (libfe_b200.so).
 *
 * Drop-in boundary for the data-parallel hot path of RyanEvanWolf/front_end.  The reference has
 * no plugin ABI of its own: the path sits behind OpenCV's virtual interfaces
 * (FeatureDetector::detect, DescriptorExtractor::compute, BFMatcher::{match,knnMatch}) and four
 * ROS services.  Each entry point below names the reference interface it replaces (file:line
 * relative to the reference repository).  All pointers are plain host pointers unless a comment
 * says "device"; the caller owns every input and output buffer and passes capacities; the library
 * never returns internal pointers (mirrors the reference, where every hop deep-copies:
 * src/StereoCamera.cpp:47,77,96,160).  No exceptions or aborts cross the boundary: every call
 * returns an fe_status and fe_last_error() gives the message.
 *
 * Threading: one fe_ctx = one device + one stream; a ctx is not thread-safe (callers serialise
 * per ctx exactly like the reference's mutex-per-detector, include/front_end/StereoCamera.hpp:76-77).
 * fe_set_detection() may be called from another thread than the one running detection; it takes
 * effect at the next frame boundary (fixes the unsynchronised write at src/live_stereo.cpp:104-115).
 */
#ifndef FE_ABI_H
#define FE_ABI_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FE_ABI_VERSION 6   /* 6: fe_set_freak, FE_DESC_FREAK, 64-byte rows through the matchers; SURF rows in fe_window_batch,
                              fe_window_update and fe_batch_landmarks, whose l_desc / r_desc became void *; fe_set_batch_detector
                              (all additive: no struct changed size, every earlier call behaves as before) */

/* ---- wire-compatible PODs ------------------------------------------------------------------ */

/* msg/kPoint.msg:1-7 (== cv::KeyPoint fields, src/front_end/utils.py:160-191).  28 bytes. */
typedef struct fe_kpoint {
    float x, y, size, angle, response;
    int32_t octave, class_id;
} fe_kpoint;

/* msg/cvMatch.msg:1-4 (== cv::DMatch, src/front_end/utils.py:193-207).  16 bytes. */
typedef struct fe_match {
    uint32_t queryIdx, trainIdx, imgIdx;
    float distance;
} fe_match;

typedef enum fe_status {
    FE_OK = 0,
    FE_ERR_BAD_ARG = -1,
    FE_ERR_CAPACITY = -2, /* an output did not fit; counts still report the required size, output
                             holds the first `cap` records in canonical order, nothing is corrupted */
    FE_ERR_CUDA = -3,
    FE_ERR_NO_DEVICE = -4, /* no CUDA device: there is NO CPU fallback */
    FE_ERR_UNSUPPORTED = -5
} fe_status;

/* Detector ring (cv::FastFeatureDetector::TYPE_*; src/live_stereo.cpp:293 uses TYPE_7_12). */
typedef enum fe_fast_type { FE_FAST_9_16 = 16, FE_FAST_7_12 = 12, FE_FAST_5_8 = 8 } fe_fast_type;

/* Descriptor kinds (src/front_end/features.py:455-461, bin/detect_node:28-51). */
typedef enum fe_desc_kind {
    FE_DESC_ORB256 = 0,          /* 32 x u8, rBRIEF-256 steered by kp.angle (ORB WTA_K=2, patch 31) */
    FE_DESC_SURF64 = 1,          /* 64 x f32,  src/surf.cpp:515-866 */
    FE_DESC_SURF128 = 2,         /* 128 x f32, SURF_EXTENDED */
    FE_DESC_BRIEF16 = 3,         /* 16 x u8, cv::BriefDescriptorExtractor(16) -- src/live_stereo.cpp:238 (see fe_set_brief_pattern) */
    FE_DESC_BRIEF32 = 4,         /* 32 x u8 */
    FE_DESC_BRIEF64 = 5,         /* 64 x u8 */
    FE_DESC_FREAK = 6            /* 64 x u8, cv::FREAK -- bin/detect_node:43-45, bin/result_ONE:25 (see fe_set_freak) */
} fe_desc_kind;

typedef enum fe_norm {
    FE_NORM_HAMMING = 6 /* cv::NORM_HAMMING */, FE_NORM_HAMMING2 = 7 /* cv::NORM_HAMMING2: ORB with WTA_K 3 / 4,
    src/StereoCamera.cpp:504-511 */, FE_NORM_L2 = 4 /* cv::NORM_L2 */
} fe_norm;

/* Context configuration.  Start from fe_default_config() (the reference's ORB defaults) and change what you need.  A
 * zero-initialised struct is also accepted: sizes, threshold and ring then take the defaults written below, while the
 * boolean / count fields (nonmax, n_features, edge_threshold, orientation) mean what they say (0 = off / none). */
typedef struct fe_config {
    int32_t device;          /* CUDA ordinal */
    int32_t max_width;       /* largest image the ctx will see (default 1920) */
    int32_t max_height;      /* (default 1200) */
    int32_t max_images;      /* batch capacity in IMAGES (2 per stereo pair; default 2) */
    int32_t max_keypoints;   /* per-image keypoint capacity, <= 65535 (default 16384) */
    int32_t fast_threshold;  /* FAST threshold t >= 1 (default 15; README.md:25-26) */
    int32_t fast_type;       /* fe_fast_type (default FE_FAST_9_16, ORB's internal detector) */
    int32_t nonmax;          /* 3x3 NMS on the FAST score (default 1) */
    int32_t n_features;      /* detector setpoint: keep the top-N by response, ties kept
                                (cv::ORB nfeatures / KeyPointsFilter::retainBest); <0 = keep all
                                (default 5000) */
    int32_t edge_threshold;  /* border filter in px (ORB edgeThreshold, default 31; 0 = none) */
    int32_t orientation;     /* 1: intensity-centroid angle (ORB detect); 0: angle = -1 (FASTX) */
    int32_t surf_upright;    /* SURF descriptors: 1 = upright (bin/detect_node:33-36), 0 = oriented */
    void *stream;            /* cudaStream_t to run on, or NULL to create a private stream */
} fe_config;

/* Matching configuration.
 * mode A (ratio):      mask -> kNN-2 -> Lowe ratio with singleton acceptance
 *                      src/StereoCamera.cpp:182-264, src/front_end/algorithm.py:825-853
 * mode B (crosscheck): BFMatcher(norm, crossCheck=true).match over ALL pairs (no mask, as OpenCV
 *                      asserts), then keep |yq - yt| <= max_dy
 *                      src/live_stereo.cpp:240,364-377, src/front_end/features.py:670,724-733 */
typedef enum fe_match_mode { FE_MATCH_RATIO = 0, FE_MATCH_CROSSCHECK = 1 } fe_match_mode;
typedef enum fe_mask_kind {
    FE_MASK_NONE = 0,
    FE_MASK_EPIPOLAR = 1,    /* |(yq + q_off) - (yt + t_off)| <= epi_threshold */
    FE_MASK_WINDOW = 2       /* |xq - xt| < win_w/2 && |yq - yt| < win_h/2 (WindowMatcher.cpp:104-128) */
} fe_mask_kind;
typedef struct fe_match_cfg {
    double ratio;            /* 0.8 -- a double, because the reference compares d0 < 0.8*d1 with a
                                double literal (StereoCamera.cpp:212) and 4 < 0.8*5 must be false */
    int32_t mode;            /* fe_match_mode */
    int32_t mask;            /* fe_mask_kind (mode A only) */
    int32_t norm;            /* fe_norm */
    float epi_threshold;     /* 2.0 in algorithm.py:690; 1.0 in StereoCamera.cpp:187 */
    float q_y_offset, t_y_offset; /* ROI offsets lroi.y / rroi.y (StereoCamera.cpp:187) */
    int32_t win_w, win_h;    /* searchRegion, 100 x 100 (WindowMatcher.cpp:32) */
    float max_dy;            /* 0.7 (mode B) ; <0 disables the post-filter */
} fe_match_cfg;

typedef struct fe_ctx fe_ctx;

/* ---- lifecycle ------------------------------------------------------------------------------- */
int32_t fe_abi_version(void);
void fe_default_config(fe_config *cfg);              /* ORB detector defaults: FAST-9_16 t=15 NMS, 5000 features, edge 31 */
int32_t fe_create(const fe_config *cfg, fe_ctx **out);
void fe_destroy(fe_ctx *ctx);
const char *fe_last_error(const fe_ctx *ctx);        /* ctx may be NULL: last fe_create error */
int32_t fe_device_count(void);

/* srv/controlDetection.srv:1-4 -- src/live_stereo.cpp:84-115, features.py:604-608,687-696.
 * Sets the FAST threshold and the setpoint (top-N); returns the new setpoint. */
int32_t fe_set_detection(fe_ctx *ctx, int32_t threshold, int32_t set_point, int32_t *new_set_point);

/* ---- primitive ops (single image) ------------------------------------------------------------ */

/* cv::FASTX / FeatureDetector::detect (src/live_stereo.cpp:293,306; src/utils.cpp:30;
 * bin/feature_node:50,62).  With cfg.orientation=1, n_features>=0 and edge_threshold=31 this is
 * cv::ORB::detect with nlevels=1 (features.py:378-387).  Output: raster order (y, then x);
 * size = 7 (FAST) or 31 (ORB mode); angle = -1 or IC angle in degrees; response = FAST score;
 * octave 0; class_id -1.  *n = number found (may exceed cap -> FE_ERR_CAPACITY). */
int32_t fe_detect(fe_ctx *ctx, const uint8_t *img, int32_t width, int32_t height, int32_t stride,
                  fe_kpoint *out, int32_t cap, int32_t *n);

/* The live nodes' detector for ONE eye of one frame: rows x cols grid over the ROI, FASTX (TYPE_7_12, NMS) per
 * cell with the cell's own threshold, optional cv::cornerSubPix(5x5, 40 it, 1e-3), cell + ROI offsets added
 * back, then one step of the per-cell setpoint controller.
 *   variant 0 = C++ node (src/live_stereo.cpp:277-352): cells = roi.w/cols x roi.h/rows inside the ROI; sub-pixel
 *               refinement on the CELL sub-image, offsets added afterwards; target = setPoint/(rows*cols) for every
 *               cell, clip [4, 80] (src/live_stereo.cpp:84-102,294-318);
 *   variant 1 = Python node (src/front_end/features.py:609-641): roi w/h are END coordinates of the slice
 *               [y : h+1, x : w+1]; refinement on the FULL image after the offsets; bottom row (row == 1) targets
 *               2 x bucket, the other rows 0.5 x bucket, clip [6, 80].
 * thresholds: rows*cols ints, row-major, in/out (updated when cfg.update != 0; the frame-to-frame dependency of
 * SURVEY.md row a2 lives in this array, so a stream must stay on one ctx).  Output: keypoints concatenated cell by
 * cell (row-major), raster order inside a cell, full-image coordinates, size 7, angle -1, response = FAST score.
 * cell_counts (optional): rows*cols detections per cell.  Needs fe_config.max_images >= rows*cols. */
typedef struct fe_grid_cfg {
    int32_t roi_x, roi_y, roi_w, roi_h;   /* lroi; roi_w <= 0: whole image */
    int32_t rows, cols;                   /* 0 -> 2 x 3 (src/live_stereo.cpp:65-66) */
    int32_t variant;                      /* 0 = C++ live node, 1 = Python gridDetector */
    int32_t fast_type;                    /* fe_fast_type, 0 -> FE_FAST_7_12 */
    int32_t set_point;                    /* srv/controlDetection.srv setPoint */
    int32_t min_threshold, max_threshold; /* 0 -> 4 (C++) / 6 (Python), 80 */
    int32_t subpix;                       /* 1: cornerSubPix */
    int32_t update;                       /* 1: run the controller step on `thresholds` */
} fe_grid_cfg;
int32_t fe_grid_detect(fe_ctx *ctx, const uint8_t *img, int32_t width, int32_t height, int32_t stride,
                       const fe_grid_cfg *cfg, int32_t *thresholds, fe_kpoint *out, int32_t cap, int32_t *n,
                       int32_t *cell_counts);

/* cv::cornerSubPix(img, pts, Size(5,5), Size(-1,-1), TermCriteria(EPS+ITER, 40, 0.001)) -- src/live_stereo.cpp:235-237,
 * 326,335; features.py:639.  Refines kps[i].(x, y) in place; every point must lie inside the image. */
int32_t fe_corner_subpix(fe_ctx *ctx, const uint8_t *img, int32_t width, int32_t height, int32_t stride,
                         fe_kpoint *kps, int32_t n);

/* cv::SURF::operator()(img, noArray(), kps, desc, useProvidedKeypoints = false) -- src/surf.cpp:896-980: the
 * Fast-Hessian detector (:462-512: box-filter Hessian pyramid, 3x3x3 non-maximum suppression, sub-sample interpolation,
 * sorted by KeypointGreater) followed by orientation + descriptor for every keypoint (:515-866), keypoints that fail are
 * removed.  This is what the services run when the detector table selects "SURF" (features.py:149-156, src/utils.cpp:36-53).
 * Output kps: x, y, size, angle (orientation, or 270 when upright), response = det(H), octave, class_id = sign of the
 * Laplacian.  desc (optional): n x 64 / 128 floats.  Parity: the CPU reference for this entry point is a restatement of
 * src/surf.cpp (no SURF binary exists to pin it). */
typedef struct fe_surf_params {
    float hessian_threshold;   /* 100 = cv::SURF default */
    int32_t n_octaves;         /* 0 -> 4 */
    int32_t n_octave_layers;   /* 0 -> 2 */
    int32_t extended;          /* 0: 64 floats, 1: 128 */
    int32_t upright;           /* 0: oriented, 1: upright */
} fe_surf_params;
int32_t fe_surf_detect_and_compute(fe_ctx *ctx, const uint8_t *img, int32_t width, int32_t height, int32_t stride,
                                   const fe_surf_params *params, fe_kpoint *kps, float *desc, int32_t cap, int32_t *n);
/* The same for a batch of n_images dense images (stride = width; n_images <= fe_config.max_images): scale space, maxima,
 * the KeypointGreater sort (src/surf.cpp:445-460,511) and the descriptors all stay on the device; kps [n_images][cap],
 * desc [n_images][cap][64 / 128] (optional), n [n_images]. */
int32_t fe_surf_detect_batch(fe_ctx *ctx, int32_t n_images, const uint8_t *imgs, int32_t width, int32_t height,
                             const fe_surf_params *params, fe_kpoint *kps, float *desc, int32_t cap, int32_t *n);

/* DescriptorExtractor::compute (bin/feature_node:54,66; features.py:721-722;
 * src/StereoCamera.cpp:89,128).  Keypoints too close to the border for the descriptor are
 * removed in place like OpenCV does (kps is compacted, *n_inout updated).  kp.angle is used
 * literally (ORB.compute on external keypoints does not recompute it -- SURVEY.md section 8c).
 * desc: n x 32 u8 (ORB256) or n x {64,128} f32, row-major, step = row bytes. */
int32_t fe_describe(fe_ctx *ctx, const uint8_t *img, int32_t width, int32_t height, int32_t stride,
                    fe_kpoint *kps, int32_t *n_inout, void *desc, int32_t desc_kind);

/* srv/windowMatching.srv:1-4 (bool reset, stereoLandmarks latestFrame -> windowStatus state) and the window of
 * WindowMatcher::newStereo (src/WindowMatcher.cpp:92-102: push_back, erase the oldest, match current against previous):
 * the STATEFUL entry.  The ctx keeps the previous frame's landmark list on the device; an update uploads only the new
 * frame (left keypoints + left descriptors [+ right descriptors]), returns its tracks against the previous frame and
 * shifts the window.  reset != 0 clears the window and returns nothing (the service's reset branch).
 *   cfg mode FE_MATCH_RATIO + FE_MASK_WINDOW : WindowMatcher.cpp:104-231 (box mask on the left coordinates, kNN-2, Lowe)
 *   cfg mode FE_MATCH_CROSSCHECK, FE_MASK_NONE: liveGraph (src/front_end/algorithm.py:1122,1160-1190) -- bf.match with
 *       crossCheck of the current vs previous LEFT descriptors and of the RIGHT descriptors (r_desc required); a track is
 *       a pair that is mutual on both sides with the same previous landmark.
 * wc (optional): window length and erase rule -- variant 0: C++ node, length = nWindow (`if size >= nWindow erase`:
 * nWindow - 1 frames stay; default 3 = `WindowMatcher slidingWindow(3)`, src/front_end_window_node.cpp:6), variant 1:
 * Python service (`if len >= length + 1: del [0]`, default length 2).  frames_in_window: window size after this update.  Tracks:
 * queryIdx = landmark of the new frame, trainIdx = landmark of the previous frame, ordered by queryIdx.
 * desc_kind FE_DESC_ORB256 / BRIEF16 / BRIEF32 (n x 32 / 16 u8 rows) with FE_NORM_HAMMING / HAMMING2, or FE_DESC_SURF64 /
 * SURF128 (n x 64 / 128 f32 rows) with FE_NORM_L2 (WindowMatcher.cpp:150-153's knnMatch, "Hamming-256 or L2-128"); every
 * frame of a window has rows of one kind: an update whose rows differ in kind (binary, SURF-64, SURF-128) from the previous
 * frame's fails with FE_ERR_BAD_ARG and leaves the window unchanged -- reset first. */
typedef struct fe_window_cfg {
    int32_t length;     /* nWindow (variant 0, <= 0 -> 3) / length (variant 1, <= 0 -> 2) */
    int32_t variant;    /* 0 = WindowMatcher.cpp, 1 = Python window service */
} fe_window_cfg;
int32_t fe_window_update(fe_ctx *ctx, int32_t reset, const fe_kpoint *l_kps, const void *l_desc, const void *r_desc, int32_t n,
                         int32_t desc_kind, const fe_match_cfg *cfg, const fe_window_cfg *wc, fe_match *tracks, int32_t cap,
                         int32_t *n_tracks, int32_t *frames_in_window);

/* cv::BriefDescriptorExtractor(bytes) -- src/live_stereo.cpp:238,359-360 (BRIEF-16 is what the live C++ node describes
 * with); cv2.xfeatures2d.BriefDescriptorExtractor_create(bytes, use_orientation) -- src/front_end/features.py:93-96,
 * bin/detect_node:28-29.  The arithmetic (integral image, 9 x 9 box-smoothed tests on a 48-px patch, 28-px border, first
 * test of a byte = its MSB) is OpenCV's; the (y1, x1, y2, x2) test tables live in OpenCV's generated_{16,32,64}.i, which
 * this library does not ship: the caller supplies the table of bytes * 8 tests (every offset in [-24, 24]).  Once set,
 * fe_describe(..., FE_DESC_BRIEF{16,32,64}) computes bytes-wide rows and fe_knn2 / fe_stereo_match / fe_window_match
 * accept them with FE_NORM_HAMMING (64-byte rows -- BRIEF-64, FREAK -- through the all-pairs 512-bit kernels).  use_orientation: rotate the offsets by kp.angle (contrib). */
int32_t fe_set_brief_pattern(fe_ctx *ctx, int32_t bytes, const int8_t *tests_y1x1y2x2, int32_t use_orientation);

/* cv2.xfeatures2d.FREAK_create(orientationNormalized, scaleNormalized, patternScale, nOctaves, selectedPairs) --
 * bin/detect_node:43-45; "FREAK" in the descriptor lists of bin/result_ONE:25, result_TWO:29, result_THREE:23.  Builds the
 * 64-scale x 256-orientation table of the 43 receptive fields as cv::FREAK::buildPattern does.  selected_pairs: 512 indices
 * into the 903 field pairs (i > j; index = i (i - 1) / 2 + j), cv::FREAK's own `selectedPairs` argument.  OpenCV's default
 * selection (FREAK_DEF_PAIRS, a table in opencv_contrib's freak.cpp) is not shipped with this library, so NULL is
 * FE_ERR_UNSUPPORTED.  Defaults of FREAK_create(): (1, 1, 22.0f, 4).  Once set, fe_describe(..., FE_DESC_FREAK) removes the
 * keypoints whose pattern leaves the image, writes the estimated orientation to kp.angle (degrees, as cv::FREAK does) and
 * returns 64-byte rows. */
int32_t fe_set_freak(fe_ctx *ctx, int32_t orientation_normalized, int32_t scale_normalized, float pattern_scale,
                     int32_t n_octaves, const int32_t *selected_pairs);

/* BFMatcher::knnMatch(q, t, k=2, mask) -- StereoCamera.cpp:199-201, WindowMatcher.cpp:150-153.
 * Raw kNN-2 rows: idx[2*i+j] (-1 when absent), dist[2*i+j]; ties -> lower train index. */
int32_t fe_knn2(fe_ctx *ctx, const fe_kpoint *q_kps, const void *q_desc, int32_t nq,
                const fe_kpoint *t_kps, const void *t_desc, int32_t nt, int32_t desc_kind,
                const fe_match_cfg *cfg, int32_t *idx, float *dist);

/* srv/stereoMatching.srv (bin/stereo_node:20-21 -> algorithm_one, algorithm.py:854-919) for mode A;
 * the live nodes' match stage (src/live_stereo.cpp:364-377) for mode B.
 * Output matches are ordered by queryIdx; queryIdx/trainIdx index the INPUT arrays, imgIdx = 0. */
int32_t fe_stereo_match(fe_ctx *ctx, const fe_kpoint *l_kps, const void *l_desc, int32_t nl,
                        const fe_kpoint *r_kps, const void *r_desc, int32_t nr, int32_t desc_kind,
                        const fe_match_cfg *cfg, fe_match *out, int32_t cap, int32_t *n);

/* WindowMatcher::newStereo matching stage (src/WindowMatcher.cpp:104-231): current frame's left
 * keypoints vs previous frame's, search-box mask + kNN-2 + Lowe ratio.  Same as fe_stereo_match
 * with mask = FE_MASK_WINDOW; provided under the reference's name. */
int32_t fe_window_match(fe_ctx *ctx, const fe_kpoint *cur_kps, const void *cur_desc, int32_t ncur,
                        const fe_kpoint *prev_kps, const void *prev_desc, int32_t nprev,
                        int32_t desc_kind, const fe_match_cfg *cfg, fe_match *out, int32_t cap,
                        int32_t *n);

/* ---- service-level ops ----------------------------------------------------------------------- */

/* srv/getStereoFeatures.srv:1-6 (bin/feature_node:24-80): detect + describe left and right.
 * Outputs per eye: kps (cap records), desc (cap rows), count.  proc_seconds[4] = lkp, ld, rkp, rd
 * stage times (bin/feature_node:27-34,72-75), measured with CUDA events.
 * desc_kind: FE_DESC_ORB256, FE_DESC_SURF64 / 128, or FE_DESC_BRIEF16 / 32 / 64 (the service's descriptor table,
 * features.py:455-461): detector.detect, then BriefDescriptorExtractor::compute with the table of fe_set_brief_pattern --
 * keypoints nearer than 28 px to the border (28 <= x < w - 28, 28 <= y < h - 28 kept, as floats) are removed after the
 * detector's top-N / Harris cut, in order; records are the detector's; rows of 16 / 32 / 64 bytes, packed.
 * FE_ERR_UNSUPPORTED without a table of that width, and for FE_DESC_FREAK. */
int32_t fe_stereo_features(fe_ctx *ctx, const uint8_t *left, const uint8_t *right, int32_t width,
                           int32_t height, int32_t stride, int32_t desc_kind,
                           fe_kpoint *l_kps, void *l_desc, int32_t *nl,
                           fe_kpoint *r_kps, void *r_desc, int32_t *nr, int32_t cap,
                           double *proc_seconds);

/* ---- batched pipeline (frame-sharded hot path; SURVEY.md section 8e) ----------------------- */

/* One call = detect + describe (the batch descriptor: ORB-256 by default) + match for n_pairs independent rectified pairs.
 * left/right: n_pairs contiguous images each (stride = width).  Outputs are fixed-capacity slabs:
 * kps[(2*p+eye)*kp_cap + i], desc[((2*p+eye)*kp_cap + i)*row], n_kps[2*p+eye], row = the descriptor's bytes (32 for
 * ORB-256 and BRIEF-32, 16 for BRIEF-16, 4 * 64 / 4 * 128 for SURF-64 / 128), rows packed like fe_describe's;
 * matches_a (mode A per cfg_a) / matches_b (mode B per cfg_b): [p*kp_cap + i], counts n_a[p], n_b[p].
 * Any output pointer may be NULL to skip its download (the work is still done on the device).
 * Host buffers should be pinned (fe_host_alloc) for full-speed async copies.  Batches of 96 pairs or
 * more are processed in chunks of 48 pairs on separate copy-in / compute / copy-out streams, so the
 * H2D of chunk k+1, the kernels of chunk k and the D2H of chunk k-1 overlap; results are identical. */
int32_t fe_pipeline_batch(fe_ctx *ctx, int32_t n_pairs, const uint8_t *left, const uint8_t *right,
                          int32_t width, int32_t height, const fe_match_cfg *cfg_a,
                          const fe_match_cfg *cfg_b, int32_t kp_cap,
                          fe_kpoint *kps, uint8_t *desc, int32_t *n_kps,
                          fe_match *matches_a, int32_t *n_a, fe_match *matches_b, int32_t *n_b);

/* The same pipeline split in three so that a caller (bench.py) can keep inputs resident in HBM:
 * upload (H2D, async + sync), run (kernels only, asynchronous on the ctx stream unless sync != 0),
 * download (D2H + sync). */
/* Selects the descriptor the batched pipeline computes: FE_DESC_ORB256 (default; Hamming matching),
 * FE_DESC_SURF64 / FE_DESC_SURF128 (bin/detect_node:33-41; L2 matching, `desc` rows are floats; keypoints the
 * SURF stage would drop (src/surf.cpp:953-978; cannot happen with edge_threshold >= 16) stay in place
 * with size = -1 in batch mode), or FE_DESC_BRIEF16 / FE_DESC_BRIEF32 (cv::BriefDescriptorExtractor, the service's other
 * descriptor; src/live_stereo.cpp:238,359-360 uses BRIEF-16):
 *  - the run uses the test table and use_orientation that fe_set_brief_pattern holds for that width when fe_batch_run /
 *    fe_pipeline_batch is called; FE_ERR_UNSUPPORTED here if no table of that width has been set;
 *  - detection is the ORB-256 batch's (FAST or ORB mode, top-N, HARRIS_SCORE, pyramid); then, as compute() after detect(),
 *    the keypoints nearer than 28 px to the border are removed, in order (n_kps = kept); records are the detector's;
 *  - matched with FE_NORM_HAMMING / FE_NORM_HAMMING2 (FE_NORM_L2 is FE_ERR_UNSUPPORTED); every batched entry point takes
 *    them (fe_batch_download, fe_pipeline_batch including its overlapped path, fe_batch_landmarks, fe_window_batch).
 * FE_DESC_BRIEF64 and FE_DESC_FREAK return FE_ERR_UNSUPPORTED: their 512-bit rows are matched by the host entry points
 * only (the batch's band and cross-check kernels read rows of at most 256 bits).  A ctx with the Fast-Hessian detector
 * (fe_set_batch_detector) returns FE_ERR_UNSUPPORTED for every kind: it describes with SURF. */
int32_t fe_set_batch_descriptor(fe_ctx *ctx, int32_t desc_kind);
/* Selects the detector of the batched pipeline (fe_batch_run, fe_pipeline_batch, and through them fe_batch_landmarks /
 * fe_window_batch).  surf == NULL: FAST / ORB per fe_config and the fe_set_orb_* calls (the default, unchanged).
 * surf != NULL: cv::SURF's Fast-Hessian detector with these parameters (src/surf.cpp:462-512), described with SURF-64 /
 * SURF-128 per surf->extended, oriented or upright per surf->upright, matched with FE_NORM_L2.  The service chain
 * getStereoFeatures(SURF, SURF) -> stereoMatching -> windowMatching (features.py:149-156, bin/feature_node:24-80) then runs
 * on the device from the images to the matches.
 *  - Keypoints: the maxima SURFInvoker keeps (src/surf.cpp:953-978; the batch never holds a size = -1 record), in RASTER
 *    order (y ascending, then x ascending, then KeypointGreater) -- not the KeypointGreater order of fe_surf_detect_batch,
 *    whose keypoints and rows they equal bit for bit as a set.  Sort by response on the host for the reference's order.
 *    Raster order lets mode A take the banded L2 kernel and mode B the exact tensor-core cross-check.
 *  - Rows: SURF-64 / SURF-128 floats in fe_batch_download, fe_pipeline_batch and fe_batch_landmarks;
 *    fe_set_batch_descriptor returns FE_ERR_UNSUPPORTED until the ctx is switched back with NULL, and a Hamming norm
 *    with such a batch is FE_ERR_UNSUPPORTED.
 *  - fe_set_orb_*, fe_set_detection and fe_config's FAST fields do not apply while the detector is selected; switching
 *    back with NULL restores them exactly (they are not changed).
 *  - fe_pipeline_batch runs upload -> run -> download for these batches (as for nlevels > 1): the scale space is one per
 *    ctx, so the two compute lanes of the overlapped path would overwrite each other's.
 *  - The scale space (Buffers group GRP_SURFDET) is allocated on first use; a FAST / ORB ctx allocates nothing for it.
 *  - An image can have more maxima than fe_config.max_keypoints: the call that synchronises (fe_batch_run with sync,
 *    fe_batch_download, fe_pipeline_batch) returns FE_ERR_CAPACITY, n_kps reports the number of maxima found, and that
 *    pair's outputs are unspecified (but in bounds).
 * Returns FE_ERR_BAD_ARG for more than 8 octaves / layers, FE_ERR_UNSUPPORTED if max_keypoints and max_height exceed the
 * raster selection's shared memory (one CTA per image: 2.1 B per keypoint + 4 B per row). */
int32_t fe_set_batch_detector(fe_ctx *ctx, const fe_surf_params *surf);
/* WindowMatcher::newStereo's data-parallel stage for a whole resident sequence (src/WindowMatcher.cpp:75-231;
 * BASELINE config 4).  Call after fe_batch_run(cfg_a = ratio mode, ...) on F consecutive stereo frames (pair f =
 * frame f).  The landmarks of frame f are its matches_a rows (every stereo match becomes a landmark, :79-85); for
 * f = 1 .. F-1, landmarks(f) are matched against landmarks(f-1): search-box mask on the LEFT keypoint coordinates
 * (:104-128), left descriptors (:134-148), kNN-2 (:150-153), Lowe ratio with singleton acceptance (:161-224).
 * tracks[(f-1)*cap + i] (queryIdx = landmark index in frame f, trainIdx = landmark index in frame f-1, :227-231),
 * n_tracks[f-1].  cfg: mode FE_MATCH_RATIO, mask FE_MASK_WINDOW -- or mode FE_MATCH_CROSSCHECK with FE_MASK_NONE for
 * liveGraph's tracker (src/front_end/algorithm.py:1160-1190: cross-check of the left AND of the right descriptors of
 * consecutive frames, intersected on the same previous landmark, no |dy| filter).  norm: FE_NORM_HAMMING / HAMMING2 on an
 * ORB-256 or BRIEF-16 / 32 batch, FE_NORM_L2 on a SURF-64 / SURF-128 batch (fe_set_batch_descriptor; exact FP32 distances, the liveGraph
 * mode by two all-pairs passes); a norm that does not fit the batch's descriptor is FE_ERR_UNSUPPORTED.
 * Optional triangulation (:36-51): Q = 4x4 row-major reprojection matrix, xyz[(f*cap + i)*3 .. +3] =
 * (Q [xl, yl, xl - xr, 1]^T)_{0..2} / (1000 * (.)_3) for landmark i of frame f; pass NULL, NULL to skip. */
int32_t fe_window_batch(fe_ctx *ctx, const fe_match_cfg *cfg, const double *Q, int32_t cap, fe_match *tracks,
                        int32_t *n_tracks, double *xyz);

/* cv::ORB WTA_K (features.py:378-387 sweeps 2 / 3 / 4): with 3 or 4 the descriptor holds 128 two-bit symbols (index
 * of the brightest of 3 / 4 points drawn by OpenCV's initializeOrbPattern, cv::RNG(0x12345678)) and is matched with
 * FE_NORM_HAMMING2 (differing symbols), like src/StereoCamera.cpp:504-511 selects the norm. */
int32_t fe_set_orb_wta_k(fe_ctx *ctx, int32_t wta_k);

/* cv::ORB scoreType -- the `score` field of the front_end/setDetector service (src/StereoCamera.cpp:445,462,
 * src/utils.cpp:86-90; features.py:297 lists both).  1 = FAST_SCORE (default here, what the reference's tables select);
 * 0 = HARRIS_SCORE (cv::ORB's own default): every level keeps the 2N best FAST corners, scores them with
 * HarrisResponses(blockSize 7, k 0.04) and keeps the N best by that score, ties kept; kp.response = Harris score. */
int32_t fe_set_orb_score_type(fe_ctx *ctx, int32_t score_type);

/* cv::ORB's pyramid: nlevels and scaleFactor of ORB_create(nfeatures, scaleFactor, nlevels, ...) (features.py:378-387
 * sweeps nLevels 2 / 4, bin/detect_node:50 uses the default 8; src/utils.cpp:84-94).  With nlevels > 1, fe_detect,
 * fe_stereo_features and the batched entry points behave like ORB::detectAndCompute: level l is the INTER_LINEAR_EXACT
 * resize of level l-1, each level keeps its share of n_features (ties kept), keypoints come back level-major with
 * pt scaled to the full image, size = 31 * scaleFactor^l and octave = l.  Matching is unchanged (the keypoints are
 * no longer in raster order, so masked kNN-2 uses the all-pairs kernel). */
int32_t fe_set_orb_pyramid(fe_ctx *ctx, int32_t nlevels, float scale_factor);

/* cv::ORB::setPatchSize for the rBRIEF descriptor (bin/detect_node:50-51 uses ORB_create() + setPatchSize(70) to
 * describe FAST keypoints; src/front_end/features.py:292-352 sweeps 10/30/50/70).  31 = ORB's learned
 * bit_pattern_31_; any other size uses OpenCV's makeRandomPattern(patchSize) points (cv::RNG(0x34985739)), sampled
 * with cv2's border rule (raw reflect-101 pixels outside the image).  In ORB-detect mode (fe_config.orientation = 1) the
 * intensity-centroid disc follows (radius patchSize / 2, OpenCV's umax table) and kp.size = patchSize. */
int32_t fe_set_orb_patch_size(fe_ctx *ctx, int32_t patch_size);

/* srv/stereoMatching.srv's reply for every pair of the resident batch: msg/stereoLandmarks.msg as algorithm_one packs it
 * (src/front_end/algorithm.py:893-913) -- row i of the left / right keypoint and descriptor arrays are the two ends of
 * match i, and matches[i] = {i, i, 0, distance}.  which: 0 = the ratio matches (cfg_a), 1 = the cross-check matches.
 * Slabs of `cap` rows per pair; n[p] = landmarks of pair p.  Any output pointer may be NULL.  Descriptor rows per batch
 * descriptor: 32 u8 (ORB-256, BRIEF-32), 16 u8 (BRIEF-16), 64 f32 (SURF-64), 128 f32 (SURF-128), packed (row p * cap + i). */
int32_t fe_batch_landmarks(fe_ctx *ctx, int32_t which, int32_t cap, fe_kpoint *l_kps, void *l_desc, fe_kpoint *r_kps,
                           void *r_desc, fe_match *matches, int32_t *n);

/* Pairs per chunk of fe_pipeline_batch's overlapped path (0 = the default, 48; batches of fewer than 2 chunks run
 * on the single-stream path).  A tuning knob: results do not depend on it. */
int32_t fe_set_chunk_pairs(fe_ctx *ctx, int32_t pairs);
int32_t fe_batch_upload(fe_ctx *ctx, int32_t n_pairs, const uint8_t *left, const uint8_t *right,
                        int32_t width, int32_t height);
int32_t fe_batch_run(fe_ctx *ctx, const fe_match_cfg *cfg_a, const fe_match_cfg *cfg_b, int32_t sync);
int32_t fe_batch_download(fe_ctx *ctx, int32_t kp_cap, fe_kpoint *kps, uint8_t *desc, int32_t *n_kps,
                          fe_match *matches_a, int32_t *n_a, fe_match *matches_b, int32_t *n_b);

/* ---- utilities --------------------------------------------------------------------------------- */
void *fe_host_alloc(size_t bytes);                 /* pinned host memory (cudaHostAlloc) */
void fe_host_free(void *p);
int32_t fe_sync(fe_ctx *ctx);                      /* cudaStreamSynchronize on the ctx stream */
void *fe_stream(fe_ctx *ctx);                      /* the cudaStream_t the ctx launches on */

/* Per-stage device timing (ProcTime slots, msg/ProcTime.msg).  When enabled, CUDA events bracket
 * every kernel stage of the batched pipeline; fe_stage_times returns accumulated milliseconds and
 * launch counts since the last reset.  names[i] are static strings. */
#define FE_MAX_STAGES 16
int32_t fe_profile_enable(fe_ctx *ctx, int32_t on);
int32_t fe_profile_reset(fe_ctx *ctx);
int32_t fe_stage_times(fe_ctx *ctx, int32_t cap, const char **names, double *ms, int64_t *launches,
                       int32_t *n_stages);
/* Measured issue rate of the POPC pipe (Gpopc/s) on the ctx's device: a register-only probe kernel.  This is
 * the denominator bench.py uses for the Hamming matcher's roofline (the matcher is bound by that pipe, not by
 * HBM: SURVEY.md section 8d). */
int32_t fe_measure_popc_peak(fe_ctx *ctx, double *gpopc_per_s);
/* Total kernels this ctx has launched since creation (bench.py's gpu_launches claim). */
int64_t fe_kernel_launches(const fe_ctx *ctx);
/* Bytes the batched entry points have copied host->device / device->host since creation. */
int32_t fe_transfer_bytes(const fe_ctx *ctx, int64_t *h2d, int64_t *d2h);

#ifdef __cplusplus
}
#endif
#endif /* FE_ABI_H */
