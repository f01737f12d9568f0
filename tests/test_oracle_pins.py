"""Pin the numpy oracle against (a) the committed cv2-generated golden vectors and (b) cv2's answers on
fresh inputs that this module builds (stored in golden/cv2_pins.npz by golden/make_golden_cv2_pins.py,
which calls the builders below).  CPU only.  Bar: bit-exact keypoints / responses / angles / descriptor
bits / match indices and distances."""
import numpy as np
import pytest

from conftest import golden
from oracle import fast, match, orb, synth

CV2_PINS = "cv2_pins"


def fresh_seed_pair():
    return synth.stereo_pair(300, 420, 12345)


def surf_primitive_inputs():
    """An image, square windows SURF resizes to 21 x 21 and (y, x) for fastAtan2."""
    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, (60, 80), dtype=np.uint8)
    windows = []
    # 19: FAST keypoints (size 7); 86: ORB keypoints (size 31); multiples of 21 take OpenCV's integer-decimation path
    # (ResizeAreaFast; 42 = every size-15 Fast-Hessian keypoint, 126 = size 45); the rest the general area table
    for S in (19, 86, 33, 24, 21, 20, 12, 57, 42, 63, 84, 105, 126, 147, 168, 189, 210, 231, 252, 43, 41, 125, 127):
        for rep in range(6):
            w = rng.integers(0, 256, (S, S), dtype=np.uint8)
            if rep & 1:     # few grey levels: many box sums land exactly on a rounding tie
                w = (w // 64 * 64 + rng.integers(0, 3, (S, S))).astype(np.uint8)
            windows.append(w)
    y = rng.standard_normal(2000).astype(np.float32) * 50
    x = rng.standard_normal(2000).astype(np.float32) * 50
    return img, windows, y, x


def subpix_inputs(img):
    """A small border-heavy crop, points for cornerSubPix and centres for getRectSubPix (13 x 13, partly outside)."""
    rng = np.random.default_rng(11)
    small = np.ascontiguousarray(img[40:100, 60:130])
    pts = np.stack([rng.uniform(0, 69.99, 60), rng.uniform(0, 59.99, 60)], 1).astype(np.float32)
    centres = [(float(np.float32(rng.uniform(-8, 78))), float(np.float32(rng.uniform(-8, 68)))) for _ in range(40)]
    return small, pts, centres


def harris_fresh_image():
    return synth.stereo_pair(200, 260, 77)[1]


def resize_inputs():
    rng = np.random.default_rng(0)
    out = []
    for (h, w) in ((240, 320), (123, 457), (37, 41)):
        img = rng.integers(0, 256, (h, w), dtype=np.uint8)
        out.append((img, int(np.rint(w / 1.2)), int(np.rint(h / 1.2))))
    return out


def wide_row_inputs():
    """64-byte rows clustered around 40 prototypes with planted exact duplicates, ragged counts, and the masks (epipolar band,
    window box, none) they are matched under."""
    rng = np.random.default_rng(11)
    base = rng.integers(0, 256, (40, 64), dtype=np.uint8)
    def rows(n):
        d = base[rng.integers(0, 40, n)].copy()                       # clusters: near-duplicates of 40 prototypes
        flips = rng.integers(0, 512, (n, 24))
        for i in range(n):
            for b in flips[i, :rng.integers(0, 24)]:
                d[i, b >> 3] ^= 1 << (b & 7)
        return d
    ql, tr = rows(301), rows(277)
    tr[5], tr[9], tr[100] = tr[200], tr[200], ql[17]                  # exact duplicates and an exact hit
    qx, qy = rng.uniform(0, 320, 301).astype(np.float32), np.sort(rng.integers(0, 240, 301)).astype(np.float32)
    tx, ty = rng.uniform(0, 320, 277).astype(np.float32), np.sort(rng.integers(0, 240, 277)).astype(np.float32)
    return ql, tr, (match.epipolar_mask(qy, ty, 2.0), match.window_mask(qx, qy, tx, ty, 100, 60), None)


def _assert_knn(g, p, idx, dd, cnt):
    """The oracle's knn2 against cv2's knnMatch rows, stored as per-row counts and the first `count` train indices / distances."""
    assert np.array_equal(cnt, g[p + "_knn_cnt"])
    valid = np.arange(2)[None, :] < cnt[:, None]
    assert np.array_equal(idx[valid], g[p + "_knn_idx"][valid]) and np.array_equal(dd[valid], g[p + "_knn_dist"][valid])


@pytest.mark.parametrize("ps", [16, 12, 8])
@pytest.mark.parametrize("thr", [15, 40])
@pytest.mark.parametrize("nms", [1, 0])
def test_fast_golden(ps, thr, nms):
    g = golden("fast_160x120")
    xs, ys, sc = fast.fast_detect(g["img"], thr, ps, bool(nms))
    k = "_%d_%d_%d" % (ps, thr, nms)
    assert np.array_equal(xs, g["x" + k]) and np.array_equal(ys, g["y" + k])
    assert np.array_equal(sc if nms else np.zeros_like(sc), g["r" + k])


def test_generator_is_pinned():
    g = golden("c1_640x480")
    L, R = synth.stereo_pair(480, 640, 1)
    assert np.array_equal(L, g["L"]) and np.array_equal(R, g["R"])
    g2 = golden("c2_1280x720")
    L, R = synth.stereo_pair(720, 1280, 0)
    assert int(L.astype(np.int64).sum()) == int(g2["L_sum"])
    assert int(R.astype(np.int64).sum()) == int(g2["R_sum"])


def _images(g):
    if "L" in g:
        return g["L"], g["R"]
    return synth.stereo_pair(int(g["h"]), int(g["w"]), int(g["seed"]))


@pytest.mark.parametrize("name", ["small_320x240", "c1_640x480", "c2_1280x720"])
def test_orb_golden(name):
    g = golden(name)
    for eye, img in zip("lr", _images(g)):
        r = orb.orb_detect_and_compute(img, int(g["n_features"]), int(g["fast_threshold"]))
        assert np.array_equal(r["x"], g[eye + "x"]) and np.array_equal(r["y"], g[eye + "y"])
        assert np.array_equal(r["response"], g[eye + "resp"])
        assert np.array_equal(r["angle"], g[eye + "angle"])          # bit-exact float32
        assert np.array_equal(r["desc"], g[eye + "desc"])


@pytest.mark.parametrize("name", ["small_320x240", "c1_640x480"])
def test_match_golden(name):
    g = golden(name)
    D = match.hamming_matrix(g["ldesc"], g["rdesc"])
    ly, ry = g["ly"].astype(np.float32), g["ry"].astype(np.float32)
    for thr in (1, 2):
        idx, dd, _ = match.knn2(D, match.epipolar_mask(ly, ry, float(thr)))
        assert np.array_equal(idx, g["knn_idx_%d" % thr])
        assert np.array_equal(dd, g["knn_dist_%d" % thr])
    q, t, d = match.cross_check(D)
    assert np.array_equal(q, g["cc_q"]) and np.array_equal(t, g["cc_t"]) and np.array_equal(d, g["cc_d"])


def test_window_golden():
    g = golden("window_320x240")
    D = match.hamming_matrix(g["desc1"], g["desc0"])
    idx, dd, _ = match.knn2(D, match.window_mask(g["x1"], g["y1"], g["x0"], g["y0"], 100, 100))
    assert np.array_equal(idx, g["knn_idx"]) and np.array_equal(dd, g["knn_dist"])
    q, t, d = match.window_match(np.stack([g["x1"], g["y1"]], 1), np.stack([g["x0"], g["y0"]], 1),
                                 g["desc1"], g["desc0"])
    assert len(q) > 50 and np.all(np.diff(q) > 0)


def test_l2_golden():
    g = golden("l2_300x350")
    D = match.l2_matrix(g["a"], g["b"])
    idx, dd, _ = match.knn2(D)
    assert np.array_equal(idx, g["knn_idx"])
    assert np.allclose(dd, g["knn_dist"], rtol=1e-5, atol=1e-6)
    q, t, d = match.cross_check(D)
    assert np.array_equal(q, g["cc_q"]) and np.array_equal(t, g["cc_t"])


def test_ratio_rule():
    idx = np.array([[3, 4], [5, -1], [-1, -1], [1, 2], [7, 8]], np.int32)
    dd = np.array([[8, 10], [50, np.inf], [np.inf, np.inf], [7, 10], [0, 0]], np.float32)
    q, t, d = match.lowe_ratio(idx, dd, 0.8)
    # 8 < 8.0 false; singleton accepted; empty dropped; 7 < 8 true; 0 < 0 false
    assert q.tolist() == [1, 3] and t.tolist() == [5, 1]


def test_setpoint_controller():
    thr = fast.setpoint_step([[15] * 3] * 2, [[900, 700, 833], [600, 1100, 850]], 5000)
    assert thr.tolist() == [[15, 15, 15], [14, 16, 15]]
    thr = fast.setpoint_step([[4, 80, 10]] * 2, [[0, 5000, 0]] * 2, 3000)
    assert thr.tolist() == [[4, 80, 9]] * 2
    thr = fast.setpoint_step([[6, 10, 10]] * 2, [[0, 251, 249], [0, 1001, 999]], 3000, python_variant=True)
    assert thr.tolist() == [[6, 10, 10], [6, 10, 10]]


def test_live_cv2_pin_fresh_seed():
    """The reference's call sequence through cv2 (ORB detectAndCompute, masked knnMatch, crossCheck match) on a seed that is
    not in the other fixtures."""
    g = golden(CV2_PINS)
    out = []
    for eye, img in zip("lr", fresh_seed_pair()):
        r = orb.orb_detect_and_compute(img, 800, 15)
        p = "fresh_%s_" % eye
        assert np.array_equal(r["x"], g[p + "x"]) and np.array_equal(r["y"], g[p + "y"])
        assert np.array_equal(r["angle"], g[p + "angle"]) and np.array_equal(r["desc"], g[p + "desc"])
        out.append(r)
    l, r = out
    D = match.hamming_matrix(l["desc"], r["desc"])
    _assert_knn(g, "fresh", *match.knn2(D, match.epipolar_mask(l["y"], r["y"], 2.0)))
    q, t, d = match.cross_check(D)
    assert np.array_equal(q, g["fresh_cc_q"]) and np.array_equal(t, g["fresh_cc_t"]) and np.array_equal(d, g["fresh_cc_d"])


def test_surf_primitives_pinned_against_cv2():
    """No SURF binary exists here; pin every primitive src/surf.cpp delegates to OpenCV."""
    from oracle import surf
    g = golden(CV2_PINS)
    img, windows, y, x = surf_primitive_inputs()
    assert np.array_equal(surf.integral_i32(img), g["surf_integral"])
    assert np.allclose(surf.G_ORI, g["surf_gauss13"], rtol=2e-7, atol=0)
    # the reference's own CUDA tables (src/cuda/surf.cu:537,699-721) for the two Gaussians
    assert abs(float(surf.G_ORI[6]) ** 2 - 0.02592208795249462) < 1e-8
    assert abs(float(surf.DW[9, 9]) - 0.01435048412531614) < 1e-8 and abs(float(surf.DW[0, 0]) - 3.695352233989979e-06) < 1e-11
    assert len(windows) == len(g["surf_resize21"])
    for w, want in zip(windows, g["surf_resize21"]):
        assert np.array_equal(surf.resize_area_21(w), want), w.shape[0]
    assert np.array_equal(orb.fast_atan2_deg(y, x), g["surf_atan2"])


def test_surf_oracle_properties():
    from oracle import surf
    L, R = synth.stereo_pair(120, 160, 8)
    xs, ys, _ = fast.fast_detect(L, 40, 16, True)
    m = (xs > 12) & (xs < 148) & (ys > 12) & (ys < 108)
    xs, ys = xs[m][:40], ys[m][:40]
    for ext, up in ((True, True), (False, False)):
        keep, ang, d = surf.surf_compute(L, xs, ys, np.full(len(xs), 7.0), ext, up)
        assert keep.all() and d.shape == (len(xs), 128 if ext else 64)
        assert np.allclose(np.linalg.norm(d, axis=1), 1.0, atol=1e-5)
        assert np.all(ang == 270.0) if up else np.all((ang >= 0) & (ang < 360))
    # a window hanging over the border is clamped, not dropped; an image smaller than the wavelet drops the keypoint
    keep, _, d = surf.surf_compute(L, np.array([1.0]), np.array([2.0]), np.array([7.0]), True, True)
    assert keep.all() and d.shape == (1, 128)
    keep, _, d = surf.surf_compute(L[:9, :9], np.array([4.0]), np.array([4.0]), np.array([31.0]), True, True)
    assert not keep.any() and len(d) == 0


def test_cornersubpix_pinned_against_cv2():
    """oracle/subpix.py restates cv::cornerSubPix + getRectSubPix; pinned bit-for-bit on the committed cv2 fixture
    (400 points incl. every border) and on cv2's answers for fresh points of a small image (border-heavy)."""
    from oracle import subpix
    g = golden("grid_subpix_480x360")
    img = g["img_f0_l"]
    sel = np.r_[0:160:4, 160:400:12]
    got = subpix.corner_subpix(img, g["subpix_in"][sel])
    assert np.array_equal(got, g["subpix_out"][sel])
    c2 = golden(CV2_PINS)
    small, pts, centres = subpix_inputs(img)
    assert np.array_equal(subpix.corner_subpix(small, pts), c2["subpix_small_out"])
    assert len(centres) == len(c2["subpix_rect"])
    for c, want in zip(centres, c2["subpix_rect"]):
        assert np.array_equal(subpix.rect_subpix_8u32f(small, 13, 13, c[0], c[1]), want)


@pytest.mark.parametrize("variant", ["cpp", "py"])
def test_grid_detector_golden(variant):
    """2x3 grid FAST-7_12 + per-cell controller (+ cornerSubPix on a subset) vs the reference's loops run through
    cv2: counts, responses, threshold trajectory over 3 frames exact; refined points exact."""
    from oracle import subpix
    g = golden("grid_subpix_480x360")
    roi = tuple(int(v) for v in g[variant + "_roi"])
    sp = int(g[variant + "_set_point"])
    thr = g["%s_e1_f0_thr_in" % variant]
    for f in range(3):
        img = g["img_f%d_r" % f]
        pts, resp, counts, thr = subpix.grid_detect(img, roi, thr, sp, python_variant=(variant == "py"),
                                                    subpix=(f == 0), subpix_step=211)
        want = g["%s_e1_f%d_pts" % (variant, f)]
        assert np.array_equal(counts, g["%s_e1_f%d_counts" % (variant, f)])
        assert np.array_equal(resp, g["%s_e1_f%d_resp" % (variant, f)])
        assert np.array_equal(thr, g["%s_e1_f%d_thr_out" % (variant, f)])
        if f == 0:
            sel = np.arange(0, len(want), 211)
            assert np.array_equal(pts[sel], want[sel])
            assert np.abs(pts - want).max() <= 5.0 + 1e-3      # unrefined points are within the window


@pytest.mark.parametrize("ps", [70, 50, 10])
def test_orb_patch_size_pattern_golden(ps):
    """cv::RNG + makeRandomPattern restated (oracle/orb.py) reproduce cv2.ORB(patchSize=ps).compute bit for bit on FAST
    keypoints (angle -1 used literally), including the raw reflect-101 samples outside the image (patch 70)."""
    g = golden("orbpatch_320x240")
    keep, desc = orb.orb_compute(g["img"], g["x"], g["y"], np.full(len(g["x"]), -1.0, np.float32), patch_size=ps)
    assert np.array_equal(g["x"][keep], g["p%d_x" % ps]) and np.array_equal(g["y"][keep], g["p%d_y" % ps])
    assert np.array_equal(desc, g["p%d_desc" % ps])


@pytest.mark.parametrize("tag", ["a", "b", "c"])
def test_orb_pyramid_golden(tag):
    """Multi-level ORB restated (INTER_LINEAR_EXACT pyramid from the previous level, per-level quotas with ties, scaled
    output) == cv2.ORB_create(nlevels = 3 / 4 / 8).detectAndCompute bit for bit: positions, size, octave, response,
    angle bit patterns and all 256 descriptor bits."""
    g = golden("orb_pyramid")
    n, lv = (int(v) for v in g[tag + "_params"])
    r = orb.orb_pyramid_detect_and_compute(g[tag + "_l_img"], n, lv)
    for k in ("x", "y", "octave", "size", "angle", "response", "desc"):
        assert np.array_equal(r[k], g["%s_l_%s" % (tag, k)]), k


@pytest.mark.parametrize("tag", ["a", "b", "c"])
def test_orb_harris_score_golden(tag):
    """scoreType = HARRIS_SCORE restated (2N FAST survivors per level -> HarrisResponses in float32 -> retainBest(N), ties
    kept) == cv2 bit for bit at 1 / 4 / 8 levels (c = cv2.ORB_create() defaults, as bin/detect_node:50 builds it):
    positions, octave, Harris responses as f32 bit patterns, angles, descriptors; and live against cv2 on a fresh seed."""
    g = golden("orb_harris")
    h, w, n, lv, thr, seed = (int(v) for v in g[tag + "_params"])
    img = synth.stereo_pair(h, w, seed)[0]
    if lv == 1:
        r = orb.orb_detect_and_compute(img, n, thr, harris=True)
        keys = ("x", "y", "angle", "response", "desc")
    else:
        r = orb.orb_pyramid_detect_and_compute(img, n, lv, fast_threshold=thr, harris=True)
        keys = ("x", "y", "octave", "size", "angle", "response", "desc")
    for k in keys:
        assert np.array_equal(np.asarray(r[k]).astype(g["%s_l_%s" % (tag, k)].dtype), g["%s_l_%s" % (tag, k)]), k
    if tag == "a":
        c2 = golden(CV2_PINS)
        r2 = orb.orb_detect_and_compute(harris_fresh_image(), 150, 12, harris=True)
        got = {(int(x), int(y)): v for x, y, v in zip(r2["x"], r2["y"], r2["response"])}
        assert got == {(int(x), int(y)): v for x, y, v in zip(c2["harris_x"], c2["harris_y"], c2["harris_response"])}


def test_resize_linear_exact_pinned():
    g = golden(CV2_PINS)
    for i, (img, dw, dh) in enumerate(resize_inputs()):
        assert np.array_equal(orb.resize_linear_exact(img, dw, dh), g["resize_linear_exact_%d" % i])


@pytest.mark.parametrize("k", [3, 4])
def test_orb_wta_and_hamming2_golden(k):
    """ORB WTA_K = 3 / 4 (tuple pattern from cv::RNG(0x12345678), two-bit symbols) and NORM_HAMMING2 matching restated ==
    cv2 bit for bit: descriptors, masked kNN-2 rows, cross-check matches."""
    g = golden("orb_wta_320x240")
    r = orb.orb_detect_and_compute(g["l_img"], 600, 15, wta_k=k)
    assert np.array_equal(r["x"], g["k%d_l_x" % k].astype(np.int32)) and np.array_equal(r["angle"], g["k%d_l_angle" % k])
    assert np.array_equal(r["desc"], g["k%d_l_desc" % k])
    ld, rd = g["k%d_l_desc" % k], g["k%d_r_desc" % k]
    D = match.hamming2_matrix(ld, rd)
    idx, dd, _ = match.knn2(D, match.epipolar_mask(g["k%d_l_y" % k], g["k%d_r_y" % k], 2.0))
    assert np.array_equal(idx, g["k%d_knn_idx" % k]) and np.array_equal(dd, g["k%d_knn_dist" % k])
    q, t, d = match.cross_check(D)
    assert np.array_equal(q, g["k%d_cc_q" % k]) and np.array_equal(t, g["k%d_cc_t" % k]) and np.array_equal(d, g["k%d_cc_d" % k])


def test_surf_fast_hessian_oracle_consistency():
    """The Fast-Hessian restatement (oracle/surf_detect.py, parity unpinned: no SURF binary) is at least self-consistent:
    its integral-image box responses equal an independent float64 direct summation, keypoints are strict 3x3x3 maxima above
    the threshold, sorted by the reference's KeypointGreater, and more octaves only add keypoints."""
    from oracle import surf_detect as sd
    img, _ = synth.stereo_pair(120, 160, 5)
    S = sd.integral_i32(img)
    f64 = img.astype(np.float64)
    for size in (9, 15, 27):
        det, tr = sd.layer_det_trace(S, size, 1)
        m = size // 2
        rng = np.random.default_rng(size)
        for _ in range(20):
            i, j = int(rng.integers(0, 120 - size)), int(rng.integers(0, 160 - size))

            def box(pat):
                return sum(f64[i + b:i + d, j + a:j + c].sum() * float(w) for (a, b, c, d, w) in pat)
            dx, dy, dxy = box(sd.resize_haar9(sd.DX_S, size)), box(sd.resize_haar9(sd.DY_S, size)), box(sd.resize_haar9(sd.DXY_S, size))
            # float32 box sums carry ~1e-5 absolute error each; det multiplies them
            assert abs(det[i + m, j + m] - (dx * dy - 0.81 * dxy * dxy)) <= 1e-4 * (1.0 + (abs(dx) + abs(dy) + abs(dxy)) ** 2)
            assert abs(tr[i + m, j + m] - (dx + dy)) <= 1e-4 * max(1.0, abs(dx) + abs(dy))
    k4, k2 = sd.fast_hessian(img, 100.0, 4, 2), sd.fast_hessian(img, 100.0, 2, 2)
    assert len(k4) > 50 and np.all(k4["response"] > 100.0)
    assert np.all(np.diff(k4["response"]) <= 0)
    assert len(k2) == np.sum(k4["octave"] < 2) and set(np.unique(k4["laplacian"])) <= {-1, 0, 1}


def test_brief_oracle_against_direct_box_sums():
    """oracle/brief.py (PARITY UNPINNED: no BRIEF table / binary here): the integral-image box sums equal direct 9 x 9 pixel
    sums, the border rule is 28 px, and the first test of a byte lands in its most significant bit."""
    from oracle import brief
    L, _ = synth.stereo_pair(100, 140, 4)
    xs = np.array([28.0, 27.9, 60.4, 111.0, 111.6, 70.0], np.float32)
    ys = np.array([28.0, 50.0, 40.5, 71.0, 71.9, 72.0], np.float32)
    tests = brief.random_tests(16, 3)
    keep, d = brief.brief_compute(L, xs, ys, tests)
    assert keep.tolist() == [True, False, True, True, True, False]       # x < w - 28 = 112, y < h - 28 = 72
    k = 2
    cy, cx = int(float(ys[k]) + 0.5), int(float(xs[k]) + 0.5)
    I = L.astype(np.int64)
    box = lambda y, x: I[cy + y - 4:min(cy + y + 5, 100), cx + x - 4:min(cx + x + 5, 140)].sum()
    row = d[1]
    for i in (0, 1, 7, 8, 77, 127):
        y1, x1, y2, x2 = (int(v) for v in tests[i])
        assert ((row[i // 8] >> (7 - i % 8)) & 1) == int(box(y1, x1) < box(y2, x2))


def test_freak_oracle_pattern_and_direct_means():
    """oracle/freak.py (PARITY UNPINNED: no FREAK binary / default pair table here): the pattern has the published geometry
    (43 fields: 7 staggered rings of 6 + the centre; outer radius 2/3 and sigma 1/3 of patternScale at scale 0, doubling every
    16 scales for nOctaves = 4), rotating the pattern by 256 / 6 steps permutes a ring, the integral-image means equal
    direct pixel means, the border rule and the bit layout of the SSE extraction order hold."""
    from oracle import freak
    pat = freak.Pattern(22.0, 4)
    lk = pat.lookup
    r0 = np.hypot(lk[0, 0, :, 0], lk[0, 0, :, 1])
    assert np.allclose(r0[:6], 22 * 2 / 3, rtol=1e-6) and np.allclose(r0[36:42], 22 * 2 / 24, rtol=1e-6) and r0[42] == 0
    assert np.allclose(lk[0, 0, :6, 2], 22 / 3, rtol=1e-6) and np.all(np.diff(r0[::6][:7]) < 0)
    assert np.allclose(lk[16, 0, :, :], 2 * lk[0, 0, :, :], rtol=1e-6)
    assert pat.sizes[0] == int(np.ceil(22.0)) + 1 and np.all(np.diff(pat.sizes) >= 0)
    # ring 1 is staggered by pi / 6; a rotation by 128 steps (pi) maps field k of a ring onto field k + 3
    assert np.allclose(lk[0, 128, 0:3, :2], lk[0, 0, 3:6, :2], atol=1e-5)
    assert abs(np.arctan2(lk[0, 0, 6, 1], lk[0, 0, 6, 0]) - np.pi / 6) < 1e-6
    # orientation weights: pair (0, 3) is the horizontal diameter of the outer ring
    assert pat.weights[0, 0] == int(4096.0 / (2 * 22 * 2 / 3) + 0.5) and pat.weights[0, 1] == 0
    assert pat.scale_index(7.0) == 0 and pat.scale_index(14.0) == 16 and pat.scale_index(1.0) == 0 and pat.scale_index(1e6) == 63
    L, _ = synth.stereo_pair(160, 200, 9)
    S = freak.integral_i32(L).astype(np.int64)
    kx, ky = np.float32(90.3), np.float32(71.6)
    for sc, rot, point in ((0, 0, 0), (0, 17, 5), (10, 200, 13), (20, 99, 30), (0, 3, 42), (16, 255, 41)):
        px, py, sg = lk[sc, rot, point]
        xf, yf = np.float32(px + kx), np.float32(py + ky)
        x0, y0 = int(float(np.float32(xf - sg)) + 0.5), int(float(np.float32(yf - sg)) + 0.5)
        x1, y1 = int(float(np.float32(xf + sg)) + 1.5), int(float(np.float32(yf + sg)) + 1.5)
        box = L[y0:y1, x0:x1].astype(np.int64)
        assert freak.mean_intensity(L, S, pat, kx, ky, sc, rot, point) == (box.sum() + box.size // 2) // box.size
    sel = freak.random_selection(5)
    assert len(set(sel.tolist())) == 512 and sel.max() < 903
    xs = np.array([23.0, 23.5, 100.0, 176.9, 177.0, 100.0, 100.0], np.float32)
    ys = np.array([80.0, 80.0, 23.5, 80.0, 80.0, 137.0, 60.0], np.float32)
    sz = np.array([7, 7, 7, 7, 7, 7, 14], np.float32)            # pattern sizes 23 (scale 0) and 45 (scale 16)
    keep, ang, d, val = freak.freak_compute(L, xs, ys, sz, sel, pattern=pat)
    assert keep.tolist() == [False, True, True, True, False, False, True]
    assert d.shape == (4, 64) and np.all(np.abs(ang) <= 180.0)
    for cnt in (0, 1, 15, 16, 127, 128, 300, 511):
        i, j = freak.ALL_PAIRS[sel[cnt]]
        b, u, t = cnt // 128, (cnt % 128) // 16, cnt % 16
        assert ((d[1, 16 * b + 15 - t] >> u) & 1) == int(val[1, i] >= val[1, j])
    # without orientation normalisation the angle is 0 and the values are those of the un-rotated pattern
    keep0, ang0, d0, val0 = freak.freak_compute(L, xs, ys, sz, sel, orientation_normalized=False, pattern=pat)
    assert np.all(ang0 == 0) and val0[1, 0] == freak.mean_intensity(L, S, pat, xs[2], ys[2], 0, 0, 0)
    # a bright blob to the right of the keypoint turns the estimated orientation towards it (angle ~ 0), above: ~ -90 / +90
    img = np.full((160, 200), 40, np.uint8)
    img[70:90, 110:130] = 220
    _, a, _, _ = freak.freak_compute(img, [100.0], [80.0], [7.0], sel, pattern=pat)
    assert abs(float(a[0])) < 15.0
    _, a, _, _ = freak.freak_compute(img.T.copy(), [80.0], [100.0], [7.0], sel, pattern=pat)
    assert abs(float(a[0]) - 90.0) < 15.0


def test_wide_row_matcher_pinned_against_cv2():
    """64-byte rows (BRIEF-64, FREAK): the oracle's BFMatcher restatement -- what the 512-bit GPU kernels are compared with --
    against cv2.BFMatcher(NORM_HAMMING) itself: masked kNN-2 (epipolar band and window box), the unmasked kNN-2 and crossCheck,
    on clustered rows with planted exact duplicates (first minimum wins) and ragged counts."""
    g = golden(CV2_PINS)
    ql, tr, masks = wide_row_inputs()
    D = match.hamming_matrix(ql, tr)
    assert D.max() <= 512 and D[17, 100] == 0
    for i, mask in enumerate(masks):
        idx, dd, cnt = match.knn2(D, mask)
        assert len(cnt) == len(ql)
        _assert_knn(g, "wide%d" % i, idx, dd, cnt)
    q, t, d = match.cross_check(D)
    assert len(g["wide_cc_q"]) > 20 and np.array_equal(q, g["wide_cc_q"]) and np.array_equal(t, g["wide_cc_t"])
    assert np.array_equal(d, g["wide_cc_d"])
