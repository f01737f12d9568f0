"""GPU parity tests: the CUDA path, called through the C-ABI (ctypes -> libfe_b200.so), against the
numpy oracle and the cv2-generated golden fixtures.  Bar: bit-exact keypoint sets, responses, angles,
BRIEF bits, match indices and distances (all integer / index work; the angle polynomial and blur are
float but reproduced operation by operation, so they are demanded bit-exact too -- the north-star
tolerance for orientation is 1e-3 rad).

Reference call sites being replaced are cited in include/fe_abi.h; the tests read like the calls the
reference makes: detect -> compute -> knnMatch/match -> ratio / cross-check.
"""
import numpy as np
import pytest

from conftest import golden
from oracle import fast as ofast
from oracle import match as omatch
from oracle import orb as oorb
from oracle import synth

import os as _os

ROOT_DIR = _os.path.dirname(_os.path.dirname(_os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def FE(fe):
    return fe


def _kp_tuple(k):
    return k["x"].astype(np.int32), k["y"].astype(np.int32)


# ---- a1: FAST + NMS --------------------------------------------------------------------------------
@pytest.mark.parametrize("ps", [16, 12, 8])
@pytest.mark.parametrize("thr", [15, 40])
@pytest.mark.parametrize("nms", [1, 0])
def test_fast_golden(FE, ps, thr, nms):
    g = golden("fast_160x120")
    with FE.FrontEnd(max_width=160, max_height=120, fast_threshold=thr, fast_type=ps, nonmax=bool(nms),
                     n_features=-1, edge_threshold=0, orientation=False, max_keypoints=16384) as f:
        k = f.detect(g["img"])
    key = "_%d_%d_%d" % (ps, thr, nms)
    assert np.array_equal(k["x"], g["x" + key].astype(np.float32))
    assert np.array_equal(k["y"], g["y" + key].astype(np.float32))
    assert np.array_equal(k["response"], g["r" + key].astype(np.float32))
    assert np.all(k["size"] == 7) and np.all(k["angle"] == -1) and np.all(k["octave"] == 0) and np.all(k["class_id"] == -1)


@pytest.mark.parametrize("shape", [(7, 7), (8, 9), (37, 53), (121, 333), (257, 1001), (64, 16)])
@pytest.mark.parametrize("ps", [16, 12])
def test_fast_ragged_sizes_vs_oracle(FE, shape, ps):
    h, w = shape
    rng = np.random.default_rng(h * 1000 + w)
    img = rng.integers(0, 256, size=(h, w), dtype=np.uint8)
    img[h // 3:h // 3 + 5, w // 4:w // 4 + 6] = 255     # some structure
    xs, ys, sc = ofast.fast_detect(img, 20, ps, True)
    with FE.FrontEnd(max_width=w, max_height=h, fast_threshold=20, fast_type=ps, n_features=-1,
                     edge_threshold=0, orientation=False, max_keypoints=60000) as f:
        k = f.detect(img)
    assert np.array_equal(k["x"].astype(np.int32), xs) and np.array_equal(k["y"].astype(np.int32), ys)
    assert np.array_equal(k["response"].astype(np.int32), sc)


def test_fast_strided_input_and_blank_image(FE):
    g = golden("fast_160x120")
    big = np.zeros((120, 200), np.uint8)
    big[:, :160] = g["img"]
    view = big[:, :160]                       # stride 200 != width 160
    with FE.FrontEnd(max_width=160, max_height=120, n_features=-1, edge_threshold=0, orientation=False) as f:
        import ctypes as C
        out = np.zeros(4096, FE.KPOINT)
        n = C.c_int32()
        st = f.lib.fe_detect(f.h, view.ctypes.data_as(C.c_void_p), 160, 120, 200, out.ctypes.data_as(C.c_void_p),
                             4096, C.byref(n))
        assert st == 0
        assert np.array_equal(out["x"][:n.value], g["x_16_15_1"].astype(np.float32))
        blank = np.full((120, 160), 77, np.uint8)
        assert len(f.detect(blank)) == 0


# ---- a3/a4/a5: ORB detect (top-N, IC angle) + rBRIEF ----------------------------------------------------
def _images(g):
    if "L" in g:
        return g["L"], g["R"]
    return synth.stereo_pair(int(g["h"]), int(g["w"]), int(g["seed"]))


@pytest.mark.parametrize("name", ["small_320x240", "c1_640x480", "c2_1280x720"])
def test_orb_detect_and_compute_golden(FE, name):
    g = golden(name)
    L, R = _images(g)
    h, w = L.shape
    with FE.FrontEnd(max_width=w, max_height=h, n_features=int(g["n_features"]),
                     fast_threshold=int(g["fast_threshold"])) as f:
        lk, ld, rk, rd, proc = f.stereo_features(L, R)
        for eye, k, d, img in (("l", lk, ld, L), ("r", rk, rd, R)):
            assert np.array_equal(k["x"], g[eye + "x"].astype(np.float32))
            assert np.array_equal(k["y"], g[eye + "y"].astype(np.float32))
            assert np.array_equal(k["response"], g[eye + "resp"].astype(np.float32))
            assert np.array_equal(k["angle"], g[eye + "angle"])
            assert np.all(k["size"] == 31)
            assert np.array_equal(d, g[eye + "desc"])
            # detect alone (FeatureDetector::detect) gives the same keypoints
            k2 = f.detect(img)
            assert np.array_equal(k2, k)
            # compute on supplied keypoints (DescriptorExtractor::compute) gives the same bits
            k3, d3 = f.compute(img, k)
            assert np.array_equal(k3, k) and np.array_equal(d3, d)
        assert len(proc) == 4 and all(p >= 0 for p in proc)


def test_setpoint_ties_and_control_detection(FE):
    """retainBest keeps ties (N_out >= N); controlDetection rewrites threshold + setpoint."""
    L, _ = synth.stereo_pair(240, 320, 21)
    with FE.FrontEnd(max_width=320, max_height=240, n_features=100) as f:
        for n, thr in ((100, 15), (37, 15), (300, 25), (0, 15), (100000, 10)):
            assert f.control_detection(thr, n) == n
            k = f.detect(L)
            r = oorb.orb_detect_and_compute(L, n, thr)
            assert np.array_equal(k["x"].astype(np.int32), r["x"]) and np.array_equal(k["y"].astype(np.int32), r["y"])
            assert np.array_equal(k["angle"], r["angle"])
            if 0 < n < 1000:
                assert len(k) >= n


def test_compute_removes_border_keypoints(FE):
    L, _ = synth.stereo_pair(240, 320, 22)
    kps = np.zeros(4, FE.KPOINT)
    kps["x"] = [5, 100, 315, 160]
    kps["y"] = [100, 5, 100, 120]
    kps["angle"] = [0, 10, 20, 33.5]
    with FE.FrontEnd(max_width=320, max_height=240) as f:
        k, d = f.compute(L, kps)
    assert len(k) == 1 and k["x"][0] == 160
    want = oorb.rbrief256(oorb.gaussian_blur_7x7(L), np.array([160]), np.array([120]), np.array([33.5], np.float32))
    assert np.array_equal(d, want)


# ---- a7..a10: matching ---------------------------------------------------------------------------------------
def _kps(FE, x, y):
    k = np.zeros(len(x), FE.KPOINT)
    k["x"], k["y"] = x, y
    return k


@pytest.mark.parametrize("name", ["small_320x240", "c1_640x480", "c2_1280x720"])
def test_knn_and_matching_golden(FE, name):
    g = golden(name)
    lk, rk = _kps(FE, g["lx"], g["ly"]), _kps(FE, g["rx"], g["ry"])
    ld, rd = g["ldesc"], g["rdesc"]
    with FE.FrontEnd(max_keypoints=8192) as f:
        for thr in (1, 2):
            cfg = FE.match_cfg(mask=FE.MASK_EPIPOLAR, epi_threshold=float(thr))
            idx, dist = f.knnMatch(lk, ld, rk, rd, cfg)
            assert np.array_equal(idx, g["knn_idx_%d" % thr])
            assert np.array_equal(dist, g["knn_dist_%d" % thr])
            m = f.stereo_match(lk, ld, rk, rd, cfg)
            q, t, d = omatch.lowe_ratio(g["knn_idx_%d" % thr], g["knn_dist_%d" % thr], 0.8)
            assert np.array_equal(m["queryIdx"], q) and np.array_equal(m["trainIdx"], t)
            assert np.array_equal(m["distance"], d) and np.all(m["imgIdx"] == 0)
        # mode B: crossCheck match, no |dy| filter -> the golden cv2 result
        m = f.stereo_match(lk, ld, rk, rd, FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, max_dy=-1.0))
        assert np.array_equal(m["queryIdx"], g["cc_q"]) and np.array_equal(m["trainIdx"], g["cc_t"])
        assert np.array_equal(m["distance"], g["cc_d"])
        # with the live nodes' |dy| <= 0.7 filter
        m = f.stereo_match(lk, ld, rk, rd, FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, max_dy=0.7))
        q, t, d = omatch.stereo_match_crosscheck(g["ly"], g["ry"], ld, rd, 0.7)
        assert np.array_equal(m["queryIdx"], q) and np.array_equal(m["trainIdx"], t)
        # unmasked kNN-2
        idx, dist = f.knnMatch(lk, ld, rk, rd, FE.match_cfg(mask=FE.MASK_NONE))
        oi, od, _ = omatch.knn2(omatch.hamming_matrix(ld, rd))
        assert np.array_equal(idx, oi) and np.array_equal(dist, od)


def test_roi_offsets_in_epipolar_mask(FE):
    """StereoCamera.cpp:187: |(yL + lroi.y) - (yR + rroi.y)| <= 1."""
    g = golden("small_320x240")
    lk, rk = _kps(FE, g["lx"], g["ly"]), _kps(FE, g["rx"], g["ry"])
    with FE.FrontEnd(max_keypoints=2048) as f:
        cfg = FE.match_cfg(mask=FE.MASK_EPIPOLAR, epi_threshold=1.0, q_y_offset=3.0, t_y_offset=1.0)
        idx, dist = f.knnMatch(lk, g["ldesc"], rk, g["rdesc"], cfg)
    D = omatch.hamming_matrix(g["ldesc"], g["rdesc"])
    oi, od, _ = omatch.knn2(D, omatch.epipolar_mask(g["ly"], g["ry"], 1.0, 3.0, 1.0))
    assert np.array_equal(idx, oi) and np.array_equal(dist, od)


def test_band_row_table_with_coordinates_outside_the_table(FE):
    """The banded matchers read their candidate rows from a row table of fe_config.max_height + 2 rows.  Caller-supplied
    keypoints may lie outside it (negative y, y beyond max_height, ROI offsets, sub-pixel rows, many keypoints in one row):
    the clamped rows are a superset and the ballot trim restores the exact allowed run -- results == oracle mask + kNN-2."""
    rng = np.random.default_rng(17)
    nq, nt = 700, 900
    qd = rng.integers(0, 256, size=(nq, 32), dtype=np.uint8)
    td = rng.integers(0, 256, size=(nt, 32), dtype=np.uint8)
    td[:300] = qd[rng.permutation(nq)[:300]]                     # planted matches (ties with equal rows included)
    qy = np.sort(rng.uniform(-40, 150, nq).astype(np.float32))
    ty = np.sort(np.concatenate([rng.uniform(-60, 170, nt - 200), np.full(120, 33.0), np.full(80, 64.5)]).astype(np.float32))
    qx, tx = rng.uniform(0, 300, nq).astype(np.float32), rng.uniform(0, 300, nt).astype(np.float32)
    qk, tk = _kps(FE, qx, qy), _kps(FE, tx, ty)
    D = omatch.hamming_matrix(qd, td)
    with FE.FrontEnd(max_width=320, max_height=100, max_keypoints=1024) as f:      # table rows 0 .. 101 only
        for thr, qo, to in ((2.0, 0.0, 0.0), (0.5, 0.0, 0.0), (1.0, 7.0, -3.0), (300.0, 0.0, 0.0)):
            cfg = FE.match_cfg(mask=FE.MASK_EPIPOLAR, epi_threshold=thr, q_y_offset=qo, t_y_offset=to)
            idx, dist = f.knnMatch(qk, qd, tk, td, cfg)
            oi, od, _ = omatch.knn2(D, omatch.epipolar_mask(qy, ty, thr, qo, to))
            assert np.array_equal(idx, oi) and np.array_equal(dist, od), (thr, qo, to)
        idx, dist = f.knnMatch(qk, qd, tk, td, FE.match_cfg(mask=FE.MASK_WINDOW, win_w=100, win_h=60))
        oi, od, _ = omatch.knn2(D, omatch.window_mask(qx, qy, tx, ty, 100, 60))
        assert np.array_equal(idx, oi) and np.array_equal(dist, od)
        # float descriptors through the FP32 banded kernel
        qf = rng.standard_normal((nq, 64)).astype(np.float32)
        tf = rng.standard_normal((nt, 64)).astype(np.float32)
        tf[:300] = qf[rng.permutation(nq)[:300]] + 0.05 * rng.standard_normal((300, 64)).astype(np.float32)
        cfg = FE.match_cfg(mask=FE.MASK_EPIPOLAR, epi_threshold=2.0, norm=FE.NORM_L2)
        idx, dist = f.knnMatch(qk, qf, tk, tf, cfg, kind=FE.DESC_SURF64)
        oi, od, _ = omatch.knn2(omatch.l2_matrix(qf, tf), omatch.epipolar_mask(qy, ty, 2.0))
        assert np.mean(idx == oi) >= 0.999


def test_window_match_golden(FE):
    g = golden("window_320x240")
    ck, pk = _kps(FE, g["x1"], g["y1"]), _kps(FE, g["x0"], g["y0"])
    with FE.FrontEnd(max_keypoints=2048) as f:
        idx, dist = f.knnMatch(ck, g["desc1"], pk, g["desc0"], FE.match_cfg(mask=FE.MASK_WINDOW))
        assert np.array_equal(idx, g["knn_idx"]) and np.array_equal(dist, g["knn_dist"])
        m = f.window_match(ck, g["desc1"], pk, g["desc0"])
    q, t, d = omatch.lowe_ratio(g["knn_idx"], g["knn_dist"], 0.8)
    assert np.array_equal(m["queryIdx"], q) and np.array_equal(m["trainIdx"], t) and np.array_equal(m["distance"], d)


def test_match_edge_cases(FE):
    rng = np.random.default_rng(3)
    d = rng.integers(0, 256, size=(5, 32), dtype=np.uint8)
    k = _kps(FE, np.arange(5) * 10.0, np.zeros(5))
    e = np.zeros(0, FE.KPOINT)
    ed = np.zeros((0, 32), np.uint8)
    with FE.FrontEnd(max_keypoints=64) as f:
        assert len(f.stereo_match(e, ed, k, d, FE.match_cfg())) == 0            # empty query
        assert len(f.stereo_match(k, d, e, ed, FE.match_cfg())) == 0            # empty train
        assert len(f.stereo_match(k, d, e, ed, FE.match_cfg(mode=FE.MATCH_CROSSCHECK))) == 0
        # one train row: singleton rows are accepted by the ratio rule
        m = f.stereo_match(k, d, k[:1], d[:1], FE.match_cfg(mask=FE.MASK_NONE))
        assert len(m) == 5 and np.all(m["trainIdx"] == 0)
        # identical descriptors: ties -> lowest train index; 0 < 0.8*0 is false -> nothing passes
        same = np.repeat(d[:1], 5, axis=0)
        idx, dist = f.knnMatch(k, same, k, same, FE.match_cfg(mask=FE.MASK_NONE))
        assert np.all(idx[:, 0] == 0) and np.all(idx[:, 1] == 1) and np.all(dist == 0)
        assert len(f.stereo_match(k, same, k, same, FE.match_cfg(mask=FE.MASK_NONE))) == 0
        m = f.stereo_match(k, same, k, same, FE.match_cfg(mode=FE.MATCH_CROSSCHECK, max_dy=-1))
        assert m["queryIdx"].tolist() == [0] and m["trainIdx"].tolist() == [0]
        # capacity: more keypoints than the ctx holds
        big = _kps(FE, np.zeros(65), np.zeros(65))
        with pytest.raises(FE.FeError) as err:
            f.stereo_match(big, np.zeros((65, 32), np.uint8), k, d, FE.match_cfg())
        assert err.value.code == FE.lib.FE_ERR_CAPACITY


def test_detect_capacity_reports_required_size(FE):
    import ctypes as C
    g = golden("fast_160x120")
    with FE.FrontEnd(max_width=160, max_height=120, n_features=-1, edge_threshold=0, orientation=False) as f:
        out = np.zeros(10, FE.KPOINT)
        guard = out.copy()
        n = C.c_int32()
        st = f.lib.fe_detect(f.h, g["img"].ctypes.data_as(C.c_void_p), 160, 120, 160,
                             out.ctypes.data_as(C.c_void_p), 5, C.byref(n))
        assert st == FE.lib.FE_ERR_CAPACITY and n.value == len(g["x_16_15_1"])
        assert np.array_equal(out["x"][:5], g["x_16_15_1"][:5].astype(np.float32))
        assert np.array_equal(out[5:], guard[5:])           # nothing written past cap


# ---- batched pipeline (frame-sharded hot path) ------------------------------------------------------------------
def _check_pair(FE, out, p, L, R, n_features, cap):
    cfg_thr = 2.0
    refs = [oorb.orb_detect_and_compute(im, n_features, 15) for im in (L, R)]
    for e, r in enumerate(refs):
        n = out["n_kps"][2 * p + e]
        assert n == len(r["x"])
        k = out["kps"][2 * p + e][:n]
        assert np.array_equal(k["x"].astype(np.int32), r["x"]) and np.array_equal(k["y"].astype(np.int32), r["y"])
        assert np.array_equal(k["response"].astype(np.int32), r["response"])
        assert np.array_equal(k["angle"], r["angle"])
        assert np.array_equal(out["desc"][2 * p + e][:n], r["desc"])
    l, r = refs
    q, t, d = omatch.stereo_match_ratio(l["y"], r["y"], l["desc"], r["desc"], cfg_thr, 0.8)
    ma = out["matches_a"][p][:out["n_a"][p]]
    assert np.array_equal(ma["queryIdx"], q) and np.array_equal(ma["trainIdx"], t) and np.array_equal(ma["distance"], d)
    q, t, d = omatch.stereo_match_crosscheck(l["y"], r["y"], l["desc"], r["desc"], 0.7)
    mb = out["matches_b"][p][:out["n_b"][p]]
    assert np.array_equal(mb["queryIdx"], q) and np.array_equal(mb["trainIdx"], t) and np.array_equal(mb["distance"], d)


def test_pipeline_batch_vs_oracle(FE):
    h, w, P, N = 240, 320, 9, 400
    Ls, Rs = synth.stereo_batch(h, w, P, seed0=40)
    with FE.FrontEnd(max_width=w, max_height=h, max_pairs=P, max_keypoints=2048, n_features=N) as f:
        out = f.pipeline_batch(Ls, Rs, FE.match_cfg(), FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE))
        for p in range(P):
            _check_pair(FE, out, p, Ls[p], Rs[p], N, 2048)
        assert f.kernel_launches() > 0


def test_pipeline_c1_single_pair_vs_golden(FE):
    """BASELINE config 0: 640x480, FAST thr 15, setpoint 5000, ORB-256, band match -- vs cv2 golden."""
    g = golden("c1_640x480")
    with FE.FrontEnd(max_width=640, max_height=480, max_pairs=1, max_keypoints=8192, n_features=5000) as f:
        out = f.pipeline_batch(g["L"][None], g["R"][None], FE.match_cfg(epi_threshold=2.0),
                               FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, max_dy=-1.0))
    nl, nr = out["n_kps"]
    assert np.array_equal(out["desc"][0][:nl], g["ldesc"]) and np.array_equal(out["desc"][1][:nr], g["rdesc"])
    q, t, d = omatch.lowe_ratio(g["knn_idx_2"], g["knn_dist_2"], 0.8)
    ma = out["matches_a"][0][:out["n_a"][0]]
    assert np.array_equal(ma["queryIdx"], q) and np.array_equal(ma["trainIdx"], t) and np.array_equal(ma["distance"], d)
    mb = out["matches_b"][0][:out["n_b"][0]]
    assert np.array_equal(mb["queryIdx"], g["cc_q"]) and np.array_equal(mb["trainIdx"], g["cc_t"])


def test_full_size_batch_properties(FE):
    """BASELINE config 1 size (1280x720, N=5000): size-independent properties on a batch --
    batch result == single-pair result (idempotence / shard independence), raster sortedness,
    N_out >= N with ties, matches ordered by queryIdx, mutuality of cross-check matches, and
    true-disparity recovery on the rectified synthetic pair (xL - xR = 12)."""
    h, w, P, N = 720, 1280, 6, 5000
    Ls, Rs = synth.stereo_batch(h, w, P, seed0=0, n_scenes=2)
    ca, cb = FE.match_cfg(), FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE)
    with FE.FrontEnd(max_width=w, max_height=h, max_pairs=P, max_keypoints=8192, n_features=N) as f:
        out = f.pipeline_batch(Ls, Rs, ca, cb)
        out = {k: v.copy() for k, v in out.items()}
        # the same batch in reversed order gives the reversed result (no cross-pair leakage)
        rev = f.pipeline_batch(Ls[::-1].copy(), Rs[::-1].copy(), ca, cb)
        for p in range(P):
            for e in range(2):
                n = out["n_kps"][2 * p + e]
                assert n == rev["n_kps"][2 * (P - 1 - p) + e]
                assert np.array_equal(out["kps"][2 * p + e][:n], rev["kps"][2 * (P - 1 - p) + e][:n])
                assert np.array_equal(out["desc"][2 * p + e][:n], rev["desc"][2 * (P - 1 - p) + e][:n])
            na = out["n_a"][p]
            assert na == rev["n_a"][P - 1 - p]
            assert np.array_equal(out["matches_a"][p][:na], rev["matches_a"][P - 1 - p][:na])
    for p in range(P):
        for e in range(2):
            n = out["n_kps"][2 * p + e]
            k = out["kps"][2 * p + e][:n]
            assert N <= n <= 8192
            key = k["y"].astype(np.int64) * 65536 + k["x"].astype(np.int64)
            assert np.all(np.diff(key) > 0)                               # strict raster order
            assert k["x"].min() >= 31 and k["x"].max() < w - 31 and k["y"].min() >= 31 and k["y"].max() < h - 31
            assert k["response"].min() >= 15 - 1
        na, nb = out["n_a"][p], out["n_b"][p]
        ma, mb = out["matches_a"][p][:na], out["matches_b"][p][:nb]
        assert np.all(np.diff(ma["queryIdx"].astype(np.int64)) > 0) and np.all(np.diff(mb["queryIdx"].astype(np.int64)) > 0)
        assert len(np.unique(mb["trainIdx"])) == nb                       # mutual matches are one-to-one
        lk, rk = out["kps"][2 * p], out["kps"][2 * p + 1]
        assert np.all(np.abs(lk["y"][ma["queryIdx"]] - rk["y"][ma["trainIdx"]]) <= 2.0)
        assert np.all(np.abs(lk["y"][mb["queryIdx"]] - rk["y"][mb["trainIdx"]]) <= 0.7)
        disp = lk["x"][ma["queryIdx"]] - rk["x"][ma["trainIdx"]]
        assert na > 3000 and np.mean(disp == 12.0) > 0.85
    # pair 0 is seed-0-like only in structure; check one full-size pair against the oracle exactly
    _check_pair(FE, out, 1, Ls[1], Rs[1], N, 8192)


def test_cross_check_variants_agree(FE, monkeypatch):
    """The three forms of mode B -- all-pairs kernel (FE_CROSS_PRUNE=0), band candidates + LB-scan verification
    (FE_CROSS_MIH=0), and the default with the multi-index join -- and the default at a per-image capacity above the join's
    limit (falls back to the scan) emit the same matches, equal to the oracle's BFMatcher(crossCheck) + |dy| filter."""
    L, R = synth.stereo_pair(480, 640, 5)
    want = None
    for env, cap in ((("FE_CROSS_PRUNE", "0"), 8192), (("FE_CROSS_MIH", "0"), 8192), (None, 8192), (None, 20000)):
        monkeypatch.delenv("FE_CROSS_PRUNE", raising=False)
        monkeypatch.delenv("FE_CROSS_MIH", raising=False)
        if env:
            monkeypatch.setenv(*env)
        with FE.FrontEnd(max_width=640, max_height=480, max_pairs=2, max_keypoints=cap, n_features=3000) as f:
            out = f.pipeline_batch(np.stack([L, R]), np.stack([R, L]), FE.match_cfg(),
                                   FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE))
        got = [out["matches_b"][p][:out["n_b"][p]].copy() for p in range(2)]
        if want is None:
            want = got
            k = [out["kps"][e][:out["n_kps"][e]] for e in range(2)]
            d = [out["desc"][e][:out["n_kps"][e]] for e in range(2)]
            q, t, dist = omatch.stereo_match_crosscheck(k[0]["y"], k[1]["y"], d[0], d[1], 0.7)
            assert np.array_equal(got[0]["queryIdx"], q) and np.array_equal(got[0]["trainIdx"], t) and len(q) > 1500
        for p in range(2):
            assert np.array_equal(got[p], want[p]), (env, cap, p)


def test_chunked_pipeline_equals_single_stream_path(FE):
    """fe_pipeline_batch overlaps copies and kernels chunk by chunk (here 16 pairs; default 48) for batches of
    at least two chunks; the result must equal the plain upload / run / download path bit for bit (and the oracle)."""
    h, w, P, N = 240, 320, 40, 300
    Ls, Rs = synth.stereo_batch(h, w, P, seed0=70, n_scenes=3)
    ca, cb = FE.match_cfg(), FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE)
    with FE.FrontEnd(max_width=w, max_height=h, max_pairs=P, max_keypoints=1024, n_features=N) as f:
        f.set_chunk_pairs(16)
        out = f.pipeline_batch(Ls, Rs, ca, cb)
        f.batch_upload(Ls, Rs)
        f.batch_run(ca, cb, sync=True)
        ref = f.batch_download()
        h2d, d2h = f.transfer_bytes()
        assert h2d == 2 * (2 * P * w * h) and d2h > 0
    for k in ("n_kps", "n_a", "n_b"):
        assert np.array_equal(out[k], ref[k])
    for i in range(2 * P):
        n = out["n_kps"][i]
        assert np.array_equal(out["kps"][i][:n], ref["kps"][i][:n])
        assert np.array_equal(out["desc"][i][:n], ref["desc"][i][:n])
    for p in range(P):
        assert np.array_equal(out["matches_a"][p][:out["n_a"][p]], ref["matches_a"][p][:ref["n_a"][p]])
        assert np.array_equal(out["matches_b"][p][:out["n_b"][p]], ref["matches_b"][p][:ref["n_b"][p]])
    for p in (0, 15, 16, 39):
        _check_pair(FE, out, p, Ls[p], Rs[p], N, 1024)


@pytest.mark.parametrize("kind,dim", [("DESC_SURF128", 128), ("DESC_SURF64", 64)])
def test_chunked_pipeline_surf_batches(FE, kind, dim):
    """The overlapped copy / compute path also serves SURF batches (FAST keypoints, SURF descriptors, banded L2 ratio matching
    and the tensor-core cross-check, chunk by chunk on views of the float buffers): equal to upload / run / download."""
    h, w, P, N = 240, 320, 10, 300
    Ls, Rs = synth.stereo_batch(h, w, P, seed0=170, n_scenes=3)
    ca = FE.match_cfg(mask=FE.MASK_EPIPOLAR, epi_threshold=2.0, norm=FE.NORM_L2)
    cb = FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, norm=FE.NORM_L2, max_dy=0.7)
    with FE.FrontEnd(max_width=w, max_height=h, max_pairs=P, max_keypoints=1024, n_features=N, orientation=False,
                     surf_upright=True) as f:
        f.set_batch_descriptor(getattr(FE, kind))
        f.set_chunk_pairs(3)                       # 4 chunks, the last one short
        out = f.pipeline_batch(Ls, Rs, ca, cb)
        assert out["desc"].shape[2] == dim and out["desc"].dtype == np.float32
        f.batch_upload(Ls, Rs)
        f.batch_run(ca, cb, sync=True)
        ref = f.batch_download()
    for k in ("n_kps", "n_a", "n_b"):
        assert np.array_equal(out[k], ref[k])
    assert out["n_b"].min() > 100
    for i in range(2 * P):
        n = out["n_kps"][i]
        assert np.array_equal(out["kps"][i][:n], ref["kps"][i][:n]) and np.array_equal(out["desc"][i][:n], ref["desc"][i][:n])
    for p in range(P):
        assert np.array_equal(out["matches_a"][p][:out["n_a"][p]], ref["matches_a"][p][:ref["n_a"][p]])
        assert np.array_equal(out["matches_b"][p][:out["n_b"][p]], ref["matches_b"][p][:ref["n_b"][p]])


def test_knn2_unsorted_keypoints_use_general_kernel(FE):
    """Caller-supplied keypoints in arbitrary order (not raster) must still match the oracle: the banded
    kernel is only valid for sorted trains, so the all-pairs masked kernel takes over."""
    g = golden("small_320x240")
    rng = np.random.default_rng(5)
    perm = rng.permutation(len(g["rx"]))
    lk, rk = _kps(FE, g["lx"], g["ly"]), _kps(FE, g["rx"][perm], g["ry"][perm])
    rd = g["rdesc"][perm]
    D = omatch.hamming_matrix(g["ldesc"], rd)
    with FE.FrontEnd(max_keypoints=2048) as f:
        for cfg, mask in ((FE.match_cfg(mask=FE.MASK_EPIPOLAR, epi_threshold=2.0), omatch.epipolar_mask(g["ly"], g["ry"][perm], 2.0)),
                          (FE.match_cfg(mask=FE.MASK_WINDOW, win_w=60, win_h=40),
                           omatch.window_mask(g["lx"], g["ly"], g["rx"][perm], g["ry"][perm], 60, 40))):
            idx, dist = f.knnMatch(lk, g["ldesc"], rk, rd, cfg)
            oi, od, _ = omatch.knn2(D, mask)
            assert np.array_equal(idx, oi) and np.array_equal(dist, od)


# ---- a6: SURF / SURF_EXTENDED descriptors + L2 matching ------------------------------------------------------------------
def _rel_l2(a, b):
    return np.linalg.norm(a.astype(np.float64) - b, axis=1) / np.maximum(np.linalg.norm(b.astype(np.float64), axis=1), 1e-30)


@pytest.mark.parametrize("extended,upright,size,n", [(True, True, 7.0, 300), (False, True, 7.0, 120), (True, False, 7.0, 80),
                                                   (False, False, 31.0, 40), (True, True, 31.0, 60),
                                                   # win_size 42 / 84 / 126: cv::resize's integer-decimation path
                                                   (True, True, 15.0, 80), (False, False, 15.0, 40), (True, True, 30.0, 40),
                                                   (True, False, 45.0, 30), (False, True, 45.0, 30)])
def test_surf_descriptors_vs_oracle(FE, extended, upright, size, n):
    """north-star tolerance: 1e-4 relative L2 per descriptor; orientation within 1e-3 rad.  Sizes 15 / 30 / 45 give
    win_size 42 / 84 / 126 = exact multiples of 21, where cv::resize(INTER_AREA) (src/surf.cpp:772) switches to integer
    box sums ((a+b+c+d+2)>>2 for x2); the oracle's three resize paths are pinned bit-equal to cv2.resize in
    tests/test_oracle_pins.py."""
    from oracle import surf as osurf
    L, _ = synth.stereo_pair(240, 320, 31)
    xs, ys, _ = ofast.fast_detect(L, 30, 16, True)
    sel = np.linspace(0, len(xs) - 1, n).astype(int)            # spread over the image, borders included
    kps = np.zeros(n, FE.KPOINT)
    kps["x"], kps["y"], kps["size"], kps["angle"] = xs[sel], ys[sel], size, -1
    keep, ang, want = osurf.surf_compute(L, kps["x"], kps["y"], kps["size"], extended, upright)
    kind = FE.DESC_SURF128 if extended else FE.DESC_SURF64
    with FE.FrontEnd(max_width=320, max_height=240, surf_upright=upright) as f:
        k, d = f.compute(L, kps, kind)
    assert len(k) == keep.sum() and d.shape == want.shape
    assert np.array_equal(k["x"], kps["x"][keep]) and np.array_equal(k["y"], kps["y"][keep])
    dang = np.abs(((k["angle"] - ang[keep]) + 180.0) % 360.0 - 180.0) * np.pi / 180.0
    assert dang.max() <= 1e-3
    err = _rel_l2(d, want)
    assert err.max() <= 1e-4, (err.max(), int((err > 1e-4).sum()))
    assert np.allclose(np.linalg.norm(d, axis=1), 1.0, atol=1e-5)


def test_l2_matching_golden(FE):
    """BFMatcher(NORM_L2) knnMatch / crossCheck on SURF_EXTENDED-shaped vectors vs the cv2 golden."""
    g = golden("l2_300x350")
    a, b = g["a"], g["b"]
    ka, kb = _kps(FE, np.arange(len(a)), np.zeros(len(a))), _kps(FE, np.arange(len(b)), np.zeros(len(b)))
    with FE.FrontEnd(max_keypoints=1024) as f:
        idx, dist = f.knnMatch(ka, a, kb, b, FE.match_cfg(mask=FE.MASK_NONE, norm=FE.NORM_L2), kind=FE.DESC_SURF128)
        assert np.array_equal(idx, g["knn_idx"])
        assert np.allclose(dist, g["knn_dist"], rtol=1e-5, atol=1e-6)
        m = f.stereo_match(ka, a, kb, b, FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, norm=FE.NORM_L2, max_dy=-1),
                           kind=FE.DESC_SURF128)
        assert np.array_equal(m["queryIdx"], g["cc_q"]) and np.array_equal(m["trainIdx"], g["cc_t"])
        assert np.allclose(m["distance"], g["cc_d"], rtol=1e-5, atol=1e-6)
        m = f.stereo_match(ka, a, kb, b, FE.match_cfg(mask=FE.MASK_NONE, norm=FE.NORM_L2), kind=FE.DESC_SURF128)
        q, t, d = omatch.lowe_ratio(g["knn_idx"], g["knn_dist"], 0.8)
        assert np.array_equal(m["queryIdx"], q) and np.array_equal(m["trainIdx"], t)
        # 64-d, masked
        a64, b64 = np.ascontiguousarray(a[:, :64]), np.ascontiguousarray(b[:, :64])
        ka["y"], kb["y"] = np.arange(len(a)) % 7, np.arange(len(b)) % 5
        idx, dist = f.knnMatch(ka, a64, kb, b64, FE.match_cfg(mask=FE.MASK_EPIPOLAR, epi_threshold=1.0, norm=FE.NORM_L2),
                               kind=FE.DESC_SURF64)
        oi, od, _ = omatch.knn2(omatch.l2_matrix(a64, b64), omatch.epipolar_mask(ka["y"], kb["y"], 1.0))
        assert np.array_equal(idx, oi) and np.allclose(dist, od, rtol=1e-5, atol=1e-6)


def test_surf_stereo_pipeline_c3_shape(FE):
    """BASELINE config 2 (SURF_EXTENDED 128-d on FAST keypoints, L2 stereo matching), reduced size: descriptors
    within 1e-4 relative L2 of the oracle and >= 99.9 % match agreement."""
    from oracle import surf as osurf
    L, R = synth.stereo_pair(240, 320, 33)
    with FE.FrontEnd(max_width=320, max_height=240, n_features=400, orientation=False, edge_threshold=31,
                     surf_upright=True, max_keypoints=2048) as f:
        lk, ld, rk, rd, proc = f.stereo_features(L, R, kind=FE.DESC_SURF128)
        assert ld.dtype == np.float32 and ld.shape[1] == 128 and np.all(lk["size"] == 7)
        cfg = FE.match_cfg(mask=FE.MASK_EPIPOLAR, epi_threshold=2.0, norm=FE.NORM_L2)
        m = f.stereo_match(lk, ld, rk, rd, cfg, kind=FE.DESC_SURF128)
    for img, k, d in ((L, lk, ld), (R, rk, rd)):
        keep, _, want = osurf.surf_compute(img, k["x"], k["y"], k["size"], True, True)
        assert keep.all() and _rel_l2(d, want).max() <= 1e-4
    _, _, wl = osurf.surf_compute(L, lk["x"], lk["y"], lk["size"], True, True)
    _, _, wr = osurf.surf_compute(R, rk["x"], rk["y"], rk["size"], True, True)
    q, t, dd = omatch.stereo_match_ratio(lk["y"], rk["y"], wl, wr, 2.0, 0.8, norm="l2")
    got = dict(zip(m["queryIdx"].tolist(), m["trainIdx"].tolist()))
    want = dict(zip(q.tolist(), t.tolist()))
    agree = sum(1 for k_, v in want.items() if got.get(k_) == v)
    assert agree >= 0.999 * len(want) and len(got) <= 1.001 * len(want) + 1
    assert len(want) > 100


def _clustered_vectors(dim, nq, nt, seed):
    """Unit vectors with planted near matches, exact duplicates (distance ties) and near-ties."""
    rng = np.random.default_rng(seed)
    a = rng.standard_normal((nq, dim)).astype(np.float32)
    b = rng.standard_normal((nt, dim)).astype(np.float32)
    m = min(nq, nt) * 2 // 3
    perm = rng.permutation(nq)[:m]
    b[:m] = a[perm] + 0.15 * rng.standard_normal((m, dim)).astype(np.float32)     # planted matches
    b[m:m + 40] = b[:40]                                                          # exact duplicates: ties
    b[m + 40:m + 80] = b[40:80] + np.float32(1e-4) * rng.standard_normal((40, dim)).astype(np.float32)   # near-ties
    a /= np.linalg.norm(a, axis=1, keepdims=True)
    b /= np.linalg.norm(b, axis=1, keepdims=True)
    return a, b, perm, m


@pytest.mark.parametrize("dim,kind,scale", [(128, "DESC_SURF128", 1.0), (64, "DESC_SURF64", 1.0), (128, "DESC_SURF128", 37.5)])
def test_l2_tensor_core_cross_check_is_exact(FE, dim, kind, scale, monkeypatch):
    """Cross-check + |dy| <= 0.7 on float descriptors through ONE tcgen05 GEMM + candidate verification (l2verify.cu) must be
    IDENTICAL -- indices and distance bits, ties included -- to the exhaustive evaluation of every element with the same FP32
    distance definition (FE_L2_VERIFY_SWEEP=1), equal to the all-pairs FP32 kernel (FE_L2_TENSOR=0) and agree with
    BFMatcher semantics evaluated in float64 (>= 99.9 %: the float32 / float64 rounding of exact ties).  Clustered vectors
    with planted matches, exact duplicates and 1e-4 near-ties; several 128-row tiles with a ragged last tile; a second
    scale checks the power-of-two normalisation of the fp16 operands."""
    nq, nt = 1500, 1333
    a, b, perm, m = _clustered_vectors(dim, nq, nt, 11)
    a, b = (a * np.float32(scale)).astype(np.float32), (b * np.float32(scale)).astype(np.float32)
    # rows: queries spread over y = 0 .. 299; a planted train sits on its query's row (+-0.5), the rest anywhere
    rng = np.random.default_rng(3)
    qy = np.sort(rng.integers(0, 300, nq)).astype(np.float32)
    ty = rng.integers(0, 300, nt).astype(np.float32)
    ty[:m] = qy[perm] + rng.choice(np.array([-0.5, 0.0, 0.5], np.float32), m)
    order = np.argsort(ty, kind="stable")                       # raster-ordered trains (the band kernel's precondition)
    b, ty = np.ascontiguousarray(b[order]), ty[order]
    ka, kb = _kps(FE, np.zeros(nq), qy), _kps(FE, np.zeros(nt), ty)
    K = getattr(FE, kind)
    cfg_cc = FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, norm=FE.NORM_L2, max_dy=0.7)
    res = {}
    for tensor in ("1", "0"):
        monkeypatch.setenv("FE_L2_TENSOR", tensor)
        with FE.FrontEnd(max_keypoints=2048) as f:
            res[tensor] = f.stereo_match(ka, a, kb, b, cfg_cc, kind=K)
            st = f.stage_times()
        assert (st["l2_tensor"][1] > 0) == (tensor == "1")
    assert len(res["0"]) > 500
    # (the all-pairs FP32 kernel sums the 128 squared differences in another order: last-bit differences of the distances)
    assert np.array_equal(res["1"]["queryIdx"], res["0"]["queryIdx"]) and np.array_equal(res["1"]["trainIdx"], res["0"]["trainIdx"])
    assert np.allclose(res["1"]["distance"], res["0"]["distance"], rtol=2e-6, atol=0)
    # the subprocess-free twin: the same library with the GEMM replaced by the exhaustive FP32 sweep needs a fresh process
    # (the knob is read once), so it lives in test_l2_verify_sweep_equals_tensor_path below
    oq, ot, _ = omatch.stereo_match_crosscheck(qy, ty, a, b, 0.7, norm="l2")
    got, want = set(zip(res["1"]["queryIdx"].tolist(), res["1"]["trainIdx"].tolist())), set(zip(oq.tolist(), ot.tolist()))
    assert len(got & want) >= 0.999 * len(want) and len(got - want) <= 0.001 * len(want) + 1


def test_l2_verify_sweep_equals_tensor_path(FE, tmp_path):
    """The tensor-core verification against the exhaustive evaluation of EVERY element with the same FP32 distance
    definition (FE_L2_VERIFY_SWEEP=1, read once per process -> a subprocess): bit-identical match lists."""
    import os, subprocess, sys
    script = tmp_path / "sweep.py"
    script.write_text("""
import sys, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
import front_end_b200 as FE
from test_gpu_parity import _clustered_vectors
a, b, perm, m = _clustered_vectors(128, 1500, 1333, 11)
rng = np.random.default_rng(3)
qy = np.sort(rng.integers(0, 300, 1500)).astype(np.float32)
ty = rng.integers(0, 300, 1333).astype(np.float32)
ty[:m] = qy[perm] + rng.choice(np.array([-0.5, 0.0, 0.5], np.float32), m)
order = np.argsort(ty, kind="stable")
b, ty = np.ascontiguousarray(b[order]), ty[order]
def kps(y):
    k = np.zeros(len(y), FE.KPOINT); k["y"] = y; k["size"] = 7; return k
cfg = FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, norm=FE.NORM_L2, max_dy=0.7)
with FE.FrontEnd(max_keypoints=2048) as f:
    r = f.stereo_match(kps(qy), a, kps(ty), b, cfg, kind=FE.DESC_SURF128)
np.save(sys.argv[1], r)
""" % (ROOT_DIR, os.path.join(ROOT_DIR, "tests")))
    outs = []
    for sweep in ("0", "1"):
        out = str(tmp_path / ("r%s.npy" % sweep))
        env = dict(os.environ, FE_L2_VERIFY_SWEEP=sweep, FE_L2_TENSOR="1")
        p = subprocess.run([sys.executable, str(script), out], env=env, capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-2000:]
        outs.append(np.load(out))
    assert len(outs[0]) > 500 and np.array_equal(outs[0], outs[1])


@pytest.mark.parametrize("dim,kind", [(128, "DESC_SURF128"), (64, "DESC_SURF64")])
def test_l2_unmasked_paths_vs_oracle(FE, dim, kind, monkeypatch):
    """Unmasked kNN-2 and cross-check without the |dy| filter have no band candidates to verify against: by default they run
    the exact all-pairs FP32 kernel; FE_L2_TENSOR=2 opts into the APPROXIMATE tcgen05 top-k candidates (A/B only)."""
    a, b, _, _ = _clustered_vectors(dim, 1500, 1333, 11)
    ka, kb = _kps(FE, np.zeros(len(a)), np.zeros(len(a))), _kps(FE, np.zeros(len(b)), np.zeros(len(b)))
    K = getattr(FE, kind)
    cfg_knn = FE.match_cfg(mask=FE.MASK_NONE, norm=FE.NORM_L2)
    cfg_cc = FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, norm=FE.NORM_L2, max_dy=-1)
    D = omatch.l2_matrix(a, b)
    oi, od, _ = omatch.knn2(D)
    oq, ot, _ = omatch.cross_check(D)
    for tensor in ("1", "2"):
        monkeypatch.setenv("FE_L2_TENSOR", tensor)
        with FE.FrontEnd(max_keypoints=2048) as f:
            idx, dist = f.knnMatch(ka, a, kb, b, cfg_knn, kind=K)
            cc = f.stereo_match(ka, a, kb, b, cfg_cc, kind=K)
            st = f.stage_times()
        assert (st["l2_tensor"][1] > 0) == (tensor == "2")
        assert np.mean(idx[:, 0] == oi[:, 0]) >= 0.999 and np.mean(idx[:, 1] == oi[:, 1]) >= 0.999
        same = idx == oi
        assert np.allclose(dist[same], od[same], rtol=1e-5, atol=1e-6)
        got, want = set(zip(cc["queryIdx"].tolist(), cc["trainIdx"].tolist())), set(zip(oq.tolist(), ot.tolist()))
        assert len(got & want) >= 0.999 * len(want) and len(got - want) <= 0.001 * len(want) + 1


def test_batched_surf_pipeline(FE):
    """Batched FAST + SURF_EXTENDED + L2 (band ratio via the banded kernel, cross-check via tcgen05) equals the
    per-pair service calls, and the oracle on one pair."""
    from oracle import surf as osurf
    h, w, P, N = 240, 320, 3, 300
    Ls, Rs = synth.stereo_batch(h, w, P, seed0=90, n_scenes=2)
    ca = FE.match_cfg(mask=FE.MASK_EPIPOLAR, epi_threshold=2.0, norm=FE.NORM_L2)
    cb = FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, norm=FE.NORM_L2, max_dy=0.7)
    with FE.FrontEnd(max_width=w, max_height=h, max_pairs=P, max_keypoints=1024, n_features=N, orientation=False,
                     surf_upright=True) as f:
        f.set_batch_descriptor(FE.DESC_SURF128)
        out = f.pipeline_batch(Ls, Rs, ca, cb)
        assert out["desc"].dtype == np.float32 and out["desc"].shape[2] == 128
        for p in range(P):
            lk, ld, rk, rd, _ = f.stereo_features(Ls[p], Rs[p], kind=FE.DESC_SURF128)
            nl, nr = out["n_kps"][2 * p], out["n_kps"][2 * p + 1]
            assert nl == len(lk) and nr == len(rk)
            assert np.array_equal(out["kps"][2 * p][:nl], lk) and np.array_equal(out["desc"][2 * p][:nl], ld)
            assert np.array_equal(out["desc"][2 * p + 1][:nr], rd)
            ma = f.stereo_match(lk, ld, rk, rd, ca, kind=FE.DESC_SURF128)
            mb = f.stereo_match(lk, ld, rk, rd, cb, kind=FE.DESC_SURF128)
            assert np.array_equal(out["matches_a"][p][:out["n_a"][p]], ma)
            assert np.array_equal(out["matches_b"][p][:out["n_b"][p]], mb)
    lk, rk = out["kps"][0][:out["n_kps"][0]], out["kps"][1][:out["n_kps"][1]]
    _, _, wl = osurf.surf_compute(Ls[0], lk["x"], lk["y"], lk["size"], True, True)
    _, _, wr = osurf.surf_compute(Rs[0], rk["x"], rk["y"], rk["size"], True, True)
    assert _rel_l2(out["desc"][0][:len(lk)], wl).max() <= 1e-4
    q, t, _ = omatch.stereo_match_ratio(lk["y"], rk["y"], wl, wr, 2.0, 0.8, norm="l2")
    ma = out["matches_a"][0][:out["n_a"][0]]
    got, want = dict(zip(ma["queryIdx"].tolist(), ma["trainIdx"].tolist())), dict(zip(q.tolist(), t.tolist()))
    assert sum(1 for k_, v in want.items() if got.get(k_) == v) >= 0.999 * len(want) and len(want) > 50
    q, t, _ = omatch.stereo_match_crosscheck(lk["y"], rk["y"], wl, wr, 0.7, norm="l2")
    mb = out["matches_b"][0][:out["n_b"][0]]
    got, want = dict(zip(mb["queryIdx"].tolist(), mb["trainIdx"].tolist())), dict(zip(q.tolist(), t.tolist()))
    assert sum(1 for k_, v in want.items() if got.get(k_) == v) >= 0.999 * len(want) and len(want) > 50


# ---- a2 + next row 1: 2x3 grid FAST-7_12, per-cell setpoint controller, cornerSubPix -------------------------
SUBPIX_TOL = 1e-4      # px; the only deviation from the CPU order is the lane-parallel double summation


def test_corner_subpix_vs_cv2_golden(FE):
    """fe_corner_subpix == cv2.cornerSubPix(img, pts, (5,5), (-1,-1), (EPS|COUNT, 40, 1e-3)) on 400 points that
    include every image border (replicated rows / columns, the top-row right-fill quirk, out-of-image steps)."""
    g = golden("grid_subpix_480x360")
    img, pin, want = g["img_f0_l"], g["subpix_in"], g["subpix_out"]
    kps = np.zeros(len(pin), FE.KPOINT)
    kps["x"], kps["y"] = pin[:, 0], pin[:, 1]
    with FE.FrontEnd(max_width=480, max_height=360, max_keypoints=4096) as f:
        out = f.corner_subpix(img, kps)
        got = np.stack([out["x"], out["y"]], 1)
        assert np.abs(got - want).max() <= SUBPIX_TOL
        assert np.mean(np.all(got == want, 1)) >= 0.99
        # a small, border-heavy image against the oracle
        from oracle import subpix as osub
        small = np.ascontiguousarray(img[40:100, 60:130])
        rng = np.random.default_rng(5)
        pts = np.stack([rng.uniform(0, 69.99, 300), rng.uniform(0, 59.99, 300)], 1).astype(np.float32)
        k2 = np.zeros(300, FE.KPOINT)
        k2["x"], k2["y"] = pts[:, 0], pts[:, 1]
        o2 = f.corner_subpix(small, k2)
        ref = osub.corner_subpix(small, pts)
        assert np.abs(np.stack([o2["x"], o2["y"]], 1) - ref).max() <= SUBPIX_TOL
        with pytest.raises(FE.FeError):
            k2["x"][0] = 70.0           # cv::cornerSubPix asserts the point is inside the image
            f.corner_subpix(small, k2)


@pytest.mark.parametrize("variant", ["cpp", "py"])
def test_grid_detector_vs_cv2_golden(FE, variant):
    """fe_grid_detect over 3 consecutive frames and both eyes == the reference's loops run through cv2
    (src/live_stereo.cpp:277-352 / features.py:609-641): per-cell counts, FAST scores and the controller's
    threshold trajectory exact; sub-pixel positions exact for >= 99 % of ~12k points per frame, all within 1e-4 px."""
    g = golden("grid_subpix_480x360")
    roi = tuple(int(v) for v in g[variant + "_roi"])
    sp = int(g[variant + "_set_point"])
    with FE.FrontEnd(max_width=480, max_height=360, max_pairs=3, max_keypoints=8192) as f:
        for eye, tag in ((0, "l"), (1, "r")):
            thr = g["%s_e%d_f0_thr_in" % (variant, eye)]
            for fr in range(3):
                assert np.array_equal(thr, g["%s_e%d_f%d_thr_in" % (variant, eye, fr)])
                k, counts, thr = f.grid_detect(g["img_f%d_%s" % (fr, tag)], thr, sp, roi=roi,
                                               variant=1 if variant == "py" else 0, cap=20000)
                want = g["%s_e%d_f%d_pts" % (variant, eye, fr)]
                assert np.array_equal(counts, g["%s_e%d_f%d_counts" % (variant, eye, fr)])
                assert np.array_equal(thr, g["%s_e%d_f%d_thr_out" % (variant, eye, fr)])
                assert len(k) == len(want)
                assert np.array_equal(k["response"], g["%s_e%d_f%d_resp" % (variant, eye, fr)])
                got = np.stack([k["x"], k["y"]], 1)
                assert np.abs(got - want).max() <= SUBPIX_TOL
                assert np.mean(np.all(got == want, 1)) >= 0.99
                assert np.all(k["size"] == 7) and np.all(k["angle"] == -1)


def test_grid_detector_options_and_errors(FE):
    """No refinement = integer FAST positions + offsets; update=0 leaves the thresholds; capacity and geometry
    errors are reported, not corrupted."""
    from oracle import subpix as osub
    img, _ = synth.stereo_pair(200, 300, 31)
    roi = (10, 6, 280, 190)
    with FE.FrontEnd(max_width=300, max_height=200, max_pairs=3, max_keypoints=4096) as f:
        for ps, ft in ((12, FE.FAST_7_12), (16, FE.FAST_9_16), (8, FE.FAST_5_8)):
            thr0 = np.array([[12, 20, 15], [9, 30, 15]])
            k, counts, thr = f.grid_detect(img, thr0, 600, roi=roi, fast_type=ft, subpix=False, update=False, cap=30000)
            pts, resp, c2, _ = osub.grid_detect(img, roi, thr0, 600, ps=ps, subpix=False, update=False)
            assert np.array_equal(thr, thr0) and np.array_equal(counts, c2)
            assert np.array_equal(np.stack([k["x"], k["y"]], 1), pts) and np.array_equal(k["response"], resp)
        with pytest.raises(FE.FeError) as e:
            f.grid_detect(img, thr0, 600, roi=roi, cap=10)
        assert e.value.code == FE.lib.FE_ERR_CAPACITY
        with pytest.raises(FE.FeError):
            f.grid_detect(img, thr0, 600, roi=(10, 6, 300, 190))       # ROI leaves the image
        with pytest.raises(FE.FeError):
            f.grid_detect(img, np.full((5, 5), 15), 600, rows=5, cols=5)  # 25 cells > capacity


# ---- a11 / BASELINE config 4: WindowMatcher over a 10-frame window, device resident ---------------------------
def _sequence(h, w, seed, n_frames):
    fr = synth.stereo_sequence(h, w, seed, n_frames)
    return np.stack([p[0] for p in fr]), np.stack([p[1] for p in fr])


def test_window_batch_10_frames_vs_oracle(FE):
    """fe_window_batch on a 10-frame sequence == WindowMatcher.cpp:104-231 restated by the oracle, frame pair by
    frame pair: landmarks = stereo ratio matches, box mask on left coordinates, left descriptors, kNN-2, Lowe 0.8.
    Triangulation (WindowMatcher.cpp:36-51) against numpy in double."""
    h, w, F, N = 240, 320, 10, 400
    Ls, Rs = _sequence(h, w, 41, F)
    Q = np.array([[1, 0, 0, -160.5], [0, 1, 0, -120.25], [0, 0, 0, 420.0], [0, 0, 1.0 / 0.12, 0]], np.float64)
    with FE.FrontEnd(max_width=w, max_height=h, max_pairs=F, max_keypoints=1024, n_features=N) as f:
        out = f.pipeline_batch(Ls, Rs, FE.match_cfg(), None)
        tracks, n_tr, xyz = f.window_batch(Q=Q)
        # stereoLandmarks packing (algorithm.py:893-913) of the same resident batch (before any
        # single-pair host call below reuses the context's device slots)
        pk = f.batch_landmarks(0)
        for fr in (0, 4, 9):
            m = out["matches_a"][fr][:out["n_a"][fr]]
            assert pk["n"][fr] == len(m)
            assert np.array_equal(pk["l_kps"][fr][:len(m)], out["kps"][2 * fr][m["queryIdx"]])
            assert np.array_equal(pk["r_kps"][fr][:len(m)], out["kps"][2 * fr + 1][m["trainIdx"]])
            assert np.array_equal(pk["l_desc"][fr][:len(m)], out["desc"][2 * fr][m["queryIdx"]])
            assert np.array_equal(pk["r_desc"][fr][:len(m)], out["desc"][2 * fr + 1][m["trainIdx"]])
            pm = pk["matches"][fr][:len(m)]
            assert np.array_equal(pm["queryIdx"], np.arange(len(m))) and np.array_equal(pm["trainIdx"], np.arange(len(m)))
            assert np.array_equal(pm["distance"], m["distance"]) and np.all(pm["imgIdx"] == 0)
        # the single-pair host entry point gives the same tracks
        lm = []
        for fr in range(F):
            m = out["matches_a"][fr][:out["n_a"][fr]]
            lk = out["kps"][2 * fr][m["queryIdx"]]
            rk = out["kps"][2 * fr + 1][m["trainIdx"]]
            lm.append((lk, out["desc"][2 * fr][m["queryIdx"]], rk))
        for fr in range(1, F):
            got = tracks[fr - 1][:n_tr[fr - 1]]
            cur, prev = lm[fr], lm[fr - 1]
            q, t, d = omatch.window_match(np.stack([cur[0]["x"], cur[0]["y"]], 1), np.stack([prev[0]["x"], prev[0]["y"]], 1),
                                          cur[1], prev[1])
            assert np.array_equal(got["queryIdx"], q) and np.array_equal(got["trainIdx"], t)
            assert np.array_equal(got["distance"], d) and len(q) > 100
            if fr in (1, 9):
                one = f.window_match(cur[0], cur[1], prev[0], prev[1])
                assert np.array_equal(one, got)
        for fr in (0, 5, 9):
            lk, _, rk = lm[fr]
            inp = np.stack([lk["x"].astype(np.float64), lk["y"].astype(np.float64),
                            (lk["x"] - rk["x"]).astype(np.float64), np.ones(len(lk))], 0)
            hom = Q @ inp
            want = (hom[:3] / (1000.0 * hom[3])).T
            assert np.allclose(xyz[fr][:len(lk)], want, rtol=1e-12, atol=0)


def test_window_update_stateful_and_live_graph_variant(FE):
    """srv/windowMatching.srv as a stateful C-ABI entry (fe_window_update: the previous frame's landmarks stay on the device)
    and liveGraph's tracker (algorithm.py:1160-1190: cross-check of the left AND right descriptors of consecutive frames,
    same-landmark intersection) -- per update against the oracle, the batched twin (fe_window_batch in cross-check mode)
    against the same, and the window-length / reset rules of both reference variants."""
    h, w, F, N = 240, 320, 6, 400
    Ls, Rs = _sequence(h, w, 47, F)
    with FE.FrontEnd(max_width=w, max_height=h, max_pairs=F, max_keypoints=1024, n_features=N) as f:
        out = f.pipeline_batch(Ls, Rs, FE.match_cfg(), None)
        live_cfg = FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE)
        tracks_b, n_b, _ = f.window_batch(cfg=live_cfg)                 # batched liveGraph tracker
        lm = []
        for fr in range(F):
            m = out["matches_a"][fr][:out["n_a"][fr]]
            lm.append((out["kps"][2 * fr][m["queryIdx"]], out["desc"][2 * fr][m["queryIdx"]], out["desc"][2 * fr + 1][m["trainIdx"]]))
        # WindowMatcher variant, C++ rule with nWindow = 3: at most two frames stay
        for fr in range(F):
            tr, frames = f.window_update(lm[fr][0], lm[fr][1])
            assert frames == min(fr + 1, 2)
            if fr == 0:
                assert len(tr) == 0
                continue
            q, t, d = omatch.window_match(np.stack([lm[fr][0]["x"], lm[fr][0]["y"]], 1),
                                          np.stack([lm[fr - 1][0]["x"], lm[fr - 1][0]["y"]], 1), lm[fr][1], lm[fr - 1][1])
            assert len(q) > 100 and np.array_equal(tr["queryIdx"], q) and np.array_equal(tr["trainIdx"], t)
            assert np.array_equal(tr["distance"], d)
        # reset empties the window: the next frame has nothing to match against
        tr, frames = f.window_update(reset=True)
        assert len(tr) == 0 and frames == 0
        tr, frames = f.window_update(lm[2][0], lm[2][1], length=4, variant=1)
        assert len(tr) == 0 and frames == 1
        # liveGraph variant, Python window rule (length 4 -> up to four frames stay)
        for fr in (3, 4, 5):
            tr, frames = f.window_update(lm[fr][0], lm[fr][1], lm[fr][2], cfg=live_cfg, length=4, variant=1)
            assert frames == min(fr - 1, 4)
            if fr == 3:
                continue        # the previous update carried no right descriptors
            q, t, d = omatch.live_graph_tracks(lm[fr][1], lm[fr - 1][1], lm[fr][2], lm[fr - 1][2])
            assert len(q) > 100 and np.array_equal(tr["queryIdx"], q) and np.array_equal(tr["trainIdx"], t)
            assert np.array_equal(tr["distance"], d)
        for fr in range(1, F):
            q, t, d = omatch.live_graph_tracks(lm[fr][1], lm[fr - 1][1], lm[fr][2], lm[fr - 1][2])
            got = tracks_b[fr - 1][:n_b[fr - 1]]
            assert np.array_equal(got["queryIdx"], q) and np.array_equal(got["trainIdx"], t) and np.array_equal(got["distance"], d)
        with pytest.raises(FE.FeError):
            f.window_update(lm[0][0], lm[0][1], cfg=live_cfg)           # liveGraph needs the right descriptors


def test_window_batch_full_size_properties(FE):
    """BASELINE config 4 at full size (10 frames of 1280x720, N=5000): size-independent properties -- tracks ordered by
    queryIdx, inside the 100x100 search box, and the camera translation of the synthetic sequence ((3, 1) px per frame)
    recovered by the large majority of tracks."""
    h, w, F, N = 720, 1280, 10, 5000
    Ls, Rs = _sequence(h, w, 7, F)
    with FE.FrontEnd(max_width=w, max_height=h, max_pairs=F, max_keypoints=8192, n_features=N) as f:
        out = f.pipeline_batch(Ls, Rs, FE.match_cfg(), None)
        tracks, n_tr, _ = f.window_batch()
    for fr in range(1, F):
        t = tracks[fr - 1][:n_tr[fr - 1]]
        mc, mp = out["matches_a"][fr][:out["n_a"][fr]], out["matches_a"][fr - 1][:out["n_a"][fr - 1]]
        ck, pk = out["kps"][2 * fr][mc["queryIdx"]], out["kps"][2 * (fr - 1)][mp["queryIdx"]]
        assert len(t) > 3000 and np.all(np.diff(t["queryIdx"].astype(np.int64)) > 0)
        dx, dy = ck["x"][t["queryIdx"]] - pk["x"][t["trainIdx"]], ck["y"][t["queryIdx"]] - pk["y"][t["trainIdx"]]
        assert np.all(np.abs(dx) < 50) and np.all(np.abs(dy) < 50)
        assert np.mean((dx == -3) & (dy == -1)) > 0.85


def test_window_batch_and_surf_batch_with_pyramid_keypoints(FE):
    """With fe_set_orb_pyramid(nlevels > 1) keypoints -- and therefore landmarks -- are level-major, not raster-ordered: the
    window matcher and the SURF batch must not take the banded (row-table) kernels, and the SURF window bound must follow
    the largest keypoint size (patchSize * scale^(L-1)), not the level-0 size."""
    from oracle import surf as osurf
    h, w, F, N = 240, 320, 4, 500
    Ls, Rs = _sequence(h, w, 43, F)
    with FE.FrontEnd(max_width=w, max_height=h, max_pairs=F, max_keypoints=2048, n_features=N) as f:
        f.set_pyramid(3, 1.2)
        out = f.pipeline_batch(Ls, Rs, FE.match_cfg(), None)
        tracks, n_tr, _ = f.window_batch()
    k0 = out["kps"][0][:out["n_kps"][0]]
    assert (k0["octave"] == 2).any() and (np.diff(k0["y"]) < 0).any()          # really level-major
    lm = []
    for fr in range(F):
        nl, nr = out["n_kps"][2 * fr], out["n_kps"][2 * fr + 1]
        lk, rk = out["kps"][2 * fr][:nl], out["kps"][2 * fr + 1][:nr]
        q, t, d = omatch.stereo_match_ratio(lk["y"], rk["y"], out["desc"][2 * fr][:nl], out["desc"][2 * fr + 1][:nr], 2.0, 0.8)
        m = out["matches_a"][fr][:out["n_a"][fr]]
        assert np.array_equal(m["queryIdx"], q) and np.array_equal(m["trainIdx"], t) and np.array_equal(m["distance"], d)
        lm.append((lk[q], out["desc"][2 * fr][q]))
    for fr in range(1, F):
        cur, prev = lm[fr], lm[fr - 1]
        q, t, d = omatch.window_match(np.stack([cur[0]["x"], cur[0]["y"]], 1), np.stack([prev[0]["x"], prev[0]["y"]], 1),
                                      cur[1], prev[1])
        got = tracks[fr - 1][:n_tr[fr - 1]]
        assert len(q) > 100 and np.array_equal(got["queryIdx"], q) and np.array_equal(got["trainIdx"], t)
        assert np.array_equal(got["distance"], d)
    # SURF-64 batch on ORB pyramid keypoints (sizes 31 / 37.2 / 44.64 -> windows 86 / 104 / 124: beyond the staged 88 px)
    ca = FE.match_cfg(mask=FE.MASK_EPIPOLAR, epi_threshold=2.0, norm=FE.NORM_L2)
    with FE.FrontEnd(max_width=w, max_height=h, max_pairs=2, max_keypoints=1024, n_features=300, surf_upright=True) as f:
        f.set_pyramid(3, 1.2)
        f.set_batch_descriptor(FE.DESC_SURF64)
        out = f.pipeline_batch(Ls[:2], Rs[:2], ca, None)
    nl, nr = out["n_kps"][0], out["n_kps"][1]
    lk, rk = out["kps"][0][:nl], out["kps"][1][:nr]
    assert lk["size"].max() > 44 and nl > 250
    keep, _, wl = osurf.surf_compute(Ls[0], lk["x"], lk["y"], lk["size"], False, True)
    assert keep.all() and _rel_l2(out["desc"][0][:nl], wl).max() <= 1e-4
    _, _, wr = osurf.surf_compute(Rs[0], rk["x"], rk["y"], rk["size"], False, True)
    q, t, _ = omatch.stereo_match_ratio(lk["y"], rk["y"], wl, wr, 2.0, 0.8, norm="l2")
    ma = out["matches_a"][0][:out["n_a"][0]]
    got, want = dict(zip(ma["queryIdx"].tolist(), ma["trainIdx"].tolist())), dict(zip(q.tolist(), t.tolist()))
    assert len(want) > 50 and sum(1 for k_, v in want.items() if got.get(k_) == v) >= 0.999 * len(want)
    assert len(got) <= 1.001 * len(want) + 1


def test_c2_full_pipeline_vs_cv2_golden(FE):
    """BASELINE config 2 end to end at full size: the images of the cv2 golden (regenerated from their seed, checksum
    verified) go through fe_pipeline_batch; keypoints, descriptors AND both match lists must equal what cv2 produced
    (ORB.detectAndCompute, knnMatch under the band mask + Lowe 0.8, BFMatcher(crossCheck) + |dy| <= 0.7)."""
    g = golden("c2_1280x720")
    L, R = _images(g)
    assert int(L.astype(np.int64).sum()) == int(g["L_sum"]) and int(R.astype(np.int64).sum()) == int(g["R_sum"])
    with FE.FrontEnd(max_width=1280, max_height=720, max_pairs=2, max_keypoints=8192, n_features=5000) as f:
        out = f.pipeline_batch(np.stack([L, L]), np.stack([R, R]), FE.match_cfg(),
                               FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, max_dy=0.7))
    for p in (0, 1):
        for e, eye in ((0, "l"), (1, "r")):
            n = out["n_kps"][2 * p + e]
            k = out["kps"][2 * p + e][:n]
            assert n == len(g[eye + "x"])
            assert np.array_equal(k["x"], g[eye + "x"].astype(np.float32)) and np.array_equal(k["y"], g[eye + "y"].astype(np.float32))
            assert np.array_equal(k["angle"], g[eye + "angle"]) and np.array_equal(out["desc"][2 * p + e][:n], g[eye + "desc"])
        q, t, d = omatch.lowe_ratio(g["knn_idx_2"], g["knn_dist_2"], 0.8)
        ma = out["matches_a"][p][:out["n_a"][p]]
        assert np.array_equal(ma["queryIdx"], q) and np.array_equal(ma["trainIdx"], t) and np.array_equal(ma["distance"], d)
        keep = np.abs(g["ly"][g["cc_q"]].astype(np.float32) - g["ry"][g["cc_t"]].astype(np.float32)) <= np.float32(0.7)
        mb = out["matches_b"][p][:out["n_b"][p]]
        assert np.array_equal(mb["queryIdx"], g["cc_q"][keep]) and np.array_equal(mb["trainIdx"], g["cc_t"][keep])
        assert np.array_equal(mb["distance"], g["cc_d"][keep]) and len(mb) > 4000


def test_c3_full_size_surf_through_the_tensor_path(FE):
    """BASELINE config 3 at FULL size (1280x720, N = 5000 FAST keypoints, SURF_EXTENDED, batched pipeline: tcgen05 candidates +
    exact FP32 decision): a 500-descriptor sample within 1e-4 relative L2 of the oracle, and the ratio / cross-check
    matches against BFMatcher semantics evaluated in float64 on the GPU's own 5200 x 5200 real (clustered) SURF
    descriptors, first-minimum tie-breaking included: >= 99.9 % agreement (north-star tolerance)."""
    from oracle import surf as osurf
    h, w, N = 720, 1280, 5000
    Ls, Rs = synth.stereo_batch(h, w, 2, seed0=300, n_scenes=1)
    ca = FE.match_cfg(mask=FE.MASK_EPIPOLAR, epi_threshold=2.0, norm=FE.NORM_L2)
    cb = FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, norm=FE.NORM_L2, max_dy=0.7)
    with FE.FrontEnd(max_width=w, max_height=h, max_pairs=2, max_keypoints=8192, n_features=N, orientation=False,
                     surf_upright=True) as f:
        f.set_batch_descriptor(FE.DESC_SURF128)
        f.profile(True)
        out = f.pipeline_batch(Ls, Rs, ca, cb)
        assert f.stage_times()["l2_tensor"][1] > 0              # the tcgen05 kernel really ran
    p = 1
    nl, nr = int(out["n_kps"][2 * p]), int(out["n_kps"][2 * p + 1])
    assert nl >= N and nr >= N
    lk, rk = out["kps"][2 * p][:nl], out["kps"][2 * p + 1][:nr]
    ld, rd = out["desc"][2 * p][:nl], out["desc"][2 * p + 1][:nr]
    sel = np.sort(np.random.default_rng(5).choice(nl, 500, replace=False))
    keep, _, want = osurf.surf_compute(Ls[p], lk["x"][sel], lk["y"][sel], lk["size"][sel], True, True)
    assert keep.all() and _rel_l2(ld[sel], want).max() <= 1e-4
    D = omatch.l2_matrix(ld, rd)
    idx, dd, _ = omatch.knn2(D, omatch.epipolar_mask(lk["y"], rk["y"], 2.0))
    q, t, _ = omatch.lowe_ratio(idx, dd, 0.8)
    ma = out["matches_a"][p][:out["n_a"][p]]
    got, want_m = dict(zip(ma["queryIdx"].tolist(), ma["trainIdx"].tolist())), dict(zip(q.tolist(), t.tolist()))
    assert len(want_m) > 3000
    assert sum(1 for k_, v in want_m.items() if got.get(k_) == v) >= 0.999 * len(want_m) and len(got) <= 1.001 * len(want_m) + 1
    cq, ct, _ = omatch.cross_check(D)
    keep = np.abs(lk["y"][cq] - rk["y"][ct]) <= np.float32(0.7)
    mb = out["matches_b"][p][:out["n_b"][p]]
    got, want_m = set(zip(mb["queryIdx"].tolist(), mb["trainIdx"].tolist())), set(zip(cq[keep].tolist(), ct[keep].tolist()))
    assert len(want_m) > 3000 and len(got & want_m) >= 0.999 * len(want_m) and len(got - want_m) <= 0.001 * len(want_m) + 1


def test_c4_full_size_window_tracks_vs_oracle(FE):
    """BASELINE config 4 at FULL size (10 frames of 1280x720, N = 5000): the tracks of two consecutive frame pairs exactly
    against WindowMatcher.cpp:104-231 restated by the oracle on the same landmarks (box mask, kNN-2, Lowe 0.8)."""
    h, w, F, N = 720, 1280, 10, 5000
    Ls, Rs = _sequence(h, w, 9, F)
    with FE.FrontEnd(max_width=w, max_height=h, max_pairs=F, max_keypoints=8192, n_features=N) as f:
        out = f.pipeline_batch(Ls, Rs, FE.match_cfg(), None)
        tracks, n_tr, _ = f.window_batch()
    def landmarks(fr):
        m = out["matches_a"][fr][:out["n_a"][fr]]
        return out["kps"][2 * fr][m["queryIdx"]], out["desc"][2 * fr][m["queryIdx"]]
    for fr in (1, 6):
        (ck, cd), (pk, pd) = landmarks(fr), landmarks(fr - 1)
        q, t, d = omatch.window_match(np.stack([ck["x"], ck["y"]], 1), np.stack([pk["x"], pk["y"]], 1), cd, pd)
        got = tracks[fr - 1][:n_tr[fr - 1]]
        assert len(q) > 3000 and np.array_equal(got["queryIdx"], q) and np.array_equal(got["trainIdx"], t)
        assert np.array_equal(got["distance"], d)


def test_c5_size_pair_properties_and_oracle_keypoints(FE):
    """BASELINE config 5 geometry (1920x1200, N=10000): one pair exactly against the oracle for detection +
    description, matches by properties (the numpy oracle's 10k x 10k distance matrix stays within seconds)."""
    h, w, N = 1200, 1920, 10000
    Ls, Rs = synth.stereo_batch(h, w, 2, seed0=5, n_scenes=1)
    with FE.FrontEnd(max_width=w, max_height=h, max_pairs=2, max_keypoints=16384, n_features=N) as f:
        out = f.pipeline_batch(Ls, Rs, FE.match_cfg(), FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE))
    r = oorb.orb_detect_and_compute(Ls[1], N, 15)
    n = out["n_kps"][2]
    k = out["kps"][2][:n]
    assert n == len(r["x"]) >= N
    assert np.array_equal(k["x"].astype(np.int32), r["x"]) and np.array_equal(k["y"].astype(np.int32), r["y"])
    assert np.array_equal(k["angle"], r["angle"]) and np.array_equal(out["desc"][2][:n], r["desc"])
    rr = oorb.orb_detect_and_compute(Rs[1], N, 15)
    q, t, d = omatch.stereo_match_ratio(r["y"], rr["y"], r["desc"], rr["desc"], 2.0, 0.8)
    ma = out["matches_a"][1][:out["n_a"][1]]
    assert np.array_equal(ma["queryIdx"], q) and np.array_equal(ma["trainIdx"], t) and np.array_equal(ma["distance"], d)
    q, t, d = omatch.stereo_match_crosscheck(r["y"], rr["y"], r["desc"], rr["desc"], 0.7)
    mb = out["matches_b"][1][:out["n_b"][1]]
    assert np.array_equal(mb["queryIdx"], q) and np.array_equal(mb["trainIdx"], t)
    assert len(mb) > 6000


# ---- next row 2 (part): ORB::setPatchSize != 31 (the live Python node's ORB_70 descriptor) ----------------------
@pytest.mark.parametrize("ps", [70, 50, 10])
def test_orb_patch_size_vs_cv2_golden(FE, ps):
    """FAST-7_12 keypoints described with cv2.ORB_create(); setPatchSize(ps) (bin/detect_node:50-51): bit-exact
    descriptors, same keypoints kept by the border filter."""
    g = golden("orbpatch_320x240")
    img = g["img"]
    with FE.FrontEnd(max_width=320, max_height=240, max_keypoints=8192, fast_type=FE.FAST_7_12, n_features=-1,
                     edge_threshold=31, orientation=False) as f:
        f.setPatchSize(ps)
        kps = np.zeros(len(g["x"]), FE.KPOINT)
        kps["x"], kps["y"], kps["size"], kps["angle"], kps["response"] = g["x"], g["y"], 7, -1, g["response"]
        k2, desc = f.compute(img, kps)
        assert np.array_equal(k2["x"], g["p%d_x" % ps]) and np.array_equal(k2["y"], g["p%d_y" % ps])
        assert np.array_equal(desc, g["p%d_desc" % ps])
        f.setPatchSize(31)                      # back to the learned pattern
        k3, d3 = f.compute(img, kps)
        keep, want = oorb.orb_compute(img, g["x"], g["y"], np.full(len(g["x"]), -1.0, np.float32), 31)
        assert np.array_equal(d3, want)
    with FE.FrontEnd(max_width=320, max_height=240) as f2:
        with pytest.raises(FE.FeError):
            f2.setPatchSize(1)


# ---- next row 2: multi-level ORB pyramid -----------------------------------------------------------------------------
@pytest.mark.parametrize("tag", ["a", "b", "c"])
def test_orb_pyramid_vs_cv2_golden(FE, tag):
    """getStereoFeatures with cv2.ORB_create(nlevels = 3 / 4 / 8) semantics: both eyes bit-exact against cv2 (positions
    scaled to the full image, size, octave, response, angle bit patterns, descriptors), level-major raster order."""
    g = golden("orb_pyramid")
    n, lv = (int(v) for v in g[tag + "_params"])
    L, R = g[tag + "_l_img"], g[tag + "_r_img"]
    with FE.FrontEnd(max_width=L.shape[1], max_height=L.shape[0], max_keypoints=8192, n_features=n) as f:
        f.set_pyramid(lv, 1.2)
        lk, ld, rk, rd, _ = f.stereo_features(L, R)
        for k, d, eye in ((lk, ld, "l"), (rk, rd, "r")):
            for fld in ("x", "y", "octave", "size", "angle", "response"):
                assert np.array_equal(k[fld], g["%s_%s_%s" % (tag, eye, fld)]), (eye, fld)
            assert np.array_equal(d, g["%s_%s_desc" % (tag, eye)])
        k1 = f.detect(L)
        assert np.array_equal(k1, lk)
        # matching on pyramid keypoints (level-major, not raster): batched pipeline == oracle on the same features
        out = f.pipeline_batch(L[None], R[None], FE.match_cfg(), FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE))
        assert out["n_kps"][0] == len(lk) and np.array_equal(out["desc"][0][:len(lk)], ld)
        q, t, d = omatch.stereo_match_ratio(lk["y"], rk["y"], ld, rd, 2.0, 0.8)
        ma = out["matches_a"][0][:out["n_a"][0]]
        assert np.array_equal(ma["queryIdx"], q) and np.array_equal(ma["trainIdx"], t) and np.array_equal(ma["distance"], d)
        q, t, d = omatch.stereo_match_crosscheck(lk["y"], rk["y"], ld, rd, 0.7)
        mb = out["matches_b"][0][:out["n_b"][0]]
        assert np.array_equal(mb["queryIdx"], q) and np.array_equal(mb["trainIdx"], t)
        f.set_pyramid(1)
        k0 = f.detect(L)
        assert np.all(k0["octave"] == 0) and len(k0) >= n


@pytest.mark.parametrize("tag", ["a", "b", "c"])
def test_orb_harris_score_vs_cv2_golden(FE, tag):
    """fe_set_orb_score_type(HARRIS_SCORE): cv2.ORB_create(scoreType=ORB_HARRIS_SCORE) at 1 / 4 / 8 levels (c = the plain
    cv2.ORB_create() of bin/detect_node:50), both eyes bit-exact: keypoint set, Harris responses (f32 bits), octave,
    size, angle, descriptors; switching back to FAST_SCORE restores the default detector."""
    g = golden("orb_harris")
    h, w, n, lv, thr, seed = (int(v) for v in g[tag + "_params"])
    L, R = synth.stereo_pair(h, w, seed)
    with FE.FrontEnd(max_width=w, max_height=h, max_keypoints=8192, n_features=n, fast_threshold=thr) as f:
        f.setScoreType(0)
        if lv > 1:
            f.set_pyramid(lv, 1.2)
        lk, ld, rk, rd, _ = f.stereo_features(L, R)
        for k, d, eye in ((lk, ld, "l"), (rk, rd, "r")):
            for fld in ("x", "y", "octave", "size", "angle", "response"):
                assert np.array_equal(k[fld], g["%s_%s_%s" % (tag, eye, fld)]), (eye, fld)
            assert np.array_equal(d, g["%s_%s_desc" % (tag, eye)])
        assert np.array_equal(f.detect(L), lk)
        out = f.pipeline_batch(L[None], R[None], FE.match_cfg(), None)
        assert out["n_kps"][0] == len(lk) and np.array_equal(out["kps"][0][:len(lk)], lk)
        f.setScoreType(1)
        f.set_pyramid(1)
        r = oorb.orb_detect_and_compute(L, n, thr)
        k0 = f.detect(L)
        assert np.array_equal(k0["x"].astype(np.int32), r["x"]) and np.array_equal(k0["response"], r["response"].astype(np.float32))
        with pytest.raises(FE.FeError):
            f.setScoreType(2)
        # the Harris cut needs its 2N candidates resident
        f.setScoreType(0)
        f.control_detection(thr, 5000)
        with pytest.raises(FE.FeError) as e:
            f.detect(L)
        assert e.value.code == FE.lib.FE_ERR_CAPACITY


# ---- next row 2 (rest): ORB WTA_K 3 / 4 + NORM_HAMMING2 -----------------------------------------------------------------
@pytest.mark.parametrize("k", [3, 4])
def test_orb_wta_hamming2_vs_cv2_golden(FE, k):
    """cv2.ORB_create(WTA_K=k).detectAndCompute + BFMatcher(NORM_HAMMING2): descriptors, masked kNN-2, ratio matches and
    cross-check matches bit-exact, through the service calls and through the batched pipeline."""
    g = golden("orb_wta_320x240")
    L, R = g["l_img"], g["r_img"]
    ca = FE.match_cfg(norm=FE.NORM_HAMMING2)
    cb = FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, norm=FE.NORM_HAMMING2, max_dy=-1.0)
    with FE.FrontEnd(max_width=320, max_height=240, max_pairs=5, max_keypoints=2048, n_features=600) as f:
        f.setWTA_K(k)
        lk, ld, rk, rd, _ = f.stereo_features(L, R)
        assert np.array_equal(lk["x"], g["k%d_l_x" % k]) and np.array_equal(lk["angle"], g["k%d_l_angle" % k])
        assert np.array_equal(ld, g["k%d_l_desc" % k]) and np.array_equal(rd, g["k%d_r_desc" % k])
        idx, dist = f.knnMatch(lk, ld, rk, rd, ca)
        assert np.array_equal(idx, g["k%d_knn_idx" % k]) and np.array_equal(dist, g["k%d_knn_dist" % k])
        m = f.stereo_match(lk, ld, rk, rd, cb)
        assert np.array_equal(m["queryIdx"], g["k%d_cc_q" % k]) and np.array_equal(m["trainIdx"], g["k%d_cc_t" % k])
        assert np.array_equal(m["distance"], g["k%d_cc_d" % k])
        q, t, d = omatch.lowe_ratio(g["k%d_knn_idx" % k], g["k%d_knn_dist" % k], 0.8)
        out = f.pipeline_batch(np.stack([L] * 5), np.stack([R] * 5), ca, cb)         # >= 4 pairs: the batched kernels
        for p in (0, 4):
            ma = out["matches_a"][p][:out["n_a"][p]]
            assert np.array_equal(ma["queryIdx"], q) and np.array_equal(ma["trainIdx"], t) and np.array_equal(ma["distance"], d)
            mb = out["matches_b"][p][:out["n_b"][p]]
            assert np.array_equal(mb["queryIdx"], g["k%d_cc_q" % k]) and np.array_equal(mb["trainIdx"], g["k%d_cc_t" % k])


# ---- next row 3: SURF Fast-Hessian detector (+ descriptors at its multi-scale keypoints) ---------------------------------
@pytest.mark.parametrize("upright,extended", [(False, False), (True, True)])
def test_surf_fast_hessian_vs_oracle(FE, upright, extended):
    """cv::SURF::operator()(img, mask, kps, desc): detector against the restatement of src/surf.cpp:167-512 (PARITY UNPINNED:
    no SURF binary exists) -- same keypoint set and order, positions within 1e-3 px, equal size / octave / Laplacian sign,
    response within 1e-5 relative; orientation within 1e-3 rad and descriptors within 1e-4 relative L2 on a sample that
    includes the largest keypoints (windows of hundreds of pixels, produced without staging)."""
    from oracle import surf as osurf
    from oracle import surf_detect as osd
    img, _ = synth.stereo_pair(240, 320, 5)
    want = osd.fast_hessian(img, 100.0, 4, 2)
    with FE.FrontEnd(max_width=320, max_height=240, max_keypoints=4096) as f:
        k, d = f.surf_detect_and_compute(img, 100.0, 4, 2, extended=extended, upright=upright)
    assert 500 < len(k) <= len(want)
    dropped = np.zeros(len(want), bool)
    if len(k) != len(want):
        kw_all, _, _ = osurf.surf_compute(img, want["x"], want["y"], want["size"], extended, upright)
        dropped = ~kw_all
    w2 = want[~dropped]
    assert len(k) == len(w2)
    assert np.abs(k["x"] - w2["x"]).max() <= 1e-3 and np.abs(k["y"] - w2["y"]).max() <= 1e-3
    assert np.array_equal(k["size"], w2["size"]) and np.array_equal(k["octave"], w2["octave"])
    assert np.array_equal(k["class_id"], w2["laplacian"])
    assert np.all(np.abs(k["response"] - w2["response"]) <= 1e-5 * np.abs(w2["response"]))
    assert np.mean((k["x"] == w2["x"]) & (k["y"] == w2["y"]) & (k["response"] == w2["response"])) >= 0.99
    # size 15 (the second filter size; win_size 42 -> cv::resize's x2 integer path) and 30 / 45 must be in the sample
    int_dec = np.nonzero(np.isin(w2["size"], (15.0, 30.0, 45.0)))[0]
    assert (w2["size"] == 15).sum() >= 10
    sel = np.unique(np.concatenate([np.arange(0, len(w2), max(len(w2) // 40, 1)), np.argsort(-w2["size"])[:6], int_dec[:40]]))
    assert (w2["size"][sel] == 15).sum() >= 10
    ks, an, ds = osurf.surf_compute(img, w2["x"][sel], w2["y"][sel], w2["size"][sel], extended, upright)
    assert ks.all()
    da = np.abs(k["angle"][sel] - an)
    da = np.minimum(da, 360.0 - da)
    assert da.max() <= np.degrees(1e-3)
    assert _rel_l2(d[sel], ds).max() <= 1e-4
    assert w2["size"][sel].max() >= 40            # windows well beyond the staged 88 px


def test_surf_fast_hessian_batch_equals_single_image(FE):
    """fe_surf_detect_batch (scale space, maxima, KeypointGreater rank sort and descriptors device resident for a stack of
    images, more images than one scale-space chunk) == the single-image entry point, image by image, bit for bit."""
    imgs = np.stack([synth.stereo_pair(180, 260, 60 + i)[i % 2] for i in range(10)])
    with FE.FrontEnd(max_width=260, max_height=180, max_pairs=5, max_keypoints=2048) as f:
        kb, db = f.surf_detect_batch(imgs, 150.0, 3, 2, extended=True, upright=False)
        for i in (0, 3, 8, 9):
            k1, d1 = f.surf_detect_and_compute(imgs[i], 150.0, 3, 2, extended=True, upright=False)
            assert len(k1) > 100 and np.array_equal(kb[i], k1) and np.array_equal(db[i], d1)
            r = k1["response"]
            assert np.all(r[:-1] >= r[1:])                     # KeypointGreater order


# ---- cv::BriefDescriptorExtractor (the live C++ node's descriptor, src/live_stereo.cpp:238,359-360) ----------------------
@pytest.mark.parametrize("n_bytes,orient", [(16, False), (32, False), (64, False), (16, True), (32, True)])
def test_brief_descriptors_vs_oracle(FE, n_bytes, orient):
    """BRIEF-16 / 32 / 64 with a caller-supplied test table (PARITY UNPINNED for the table: OpenCV's generated_*.i is not
    in this image): bit-exact against the restatement of features2d/src/brief.cpp -- border 28, integral image, 9 x 9 box
    tests, first test of a byte = its MSB, contrib's use_orientation rotation."""
    from oracle import brief as obrief
    L, _ = synth.stereo_pair(240, 320, 21)
    xs, ys, _ = ofast.fast_detect(L, 25, 12, True)
    n = min(len(xs), 600)
    sel = np.linspace(0, len(xs) - 1, n).astype(int)
    kps = np.zeros(n, FE.KPOINT)
    kps["x"], kps["y"], kps["size"] = xs[sel] + np.float32(0.25) * (sel % 4), ys[sel] + np.float32(0.5) * (sel % 2), 7
    kps["angle"] = (sel * 37) % 360
    tests = obrief.random_tests(n_bytes, seed=n_bytes)
    keep, want = obrief.brief_compute(L, kps["x"], kps["y"], tests, kps["angle"], orient)
    kind = {16: FE.DESC_BRIEF16, 32: FE.DESC_BRIEF32, 64: FE.DESC_BRIEF64}[n_bytes]
    with FE.FrontEnd(max_width=320, max_height=240, max_keypoints=2048) as f:
        with pytest.raises(FE.FeError):
            f.compute(L, kps, kind)                                   # no table yet
        f.set_brief_pattern(tests, orient)
        k, d = f.compute(L, kps, kind)
        assert 0 < keep.sum() < n and len(k) == keep.sum() and d.shape == want.shape
        assert np.array_equal(k["x"], kps["x"][keep]) and np.array_equal(d, want)
        if n_bytes <= 32 and not orient:
            # the live node's matcher on these rows: BFMatcher(NORM_HAMMING, crossCheck) + |dy| <= 0.7
            R = synth.stereo_pair(240, 320, 21)[1]
            kr = kps.copy()
            kr["x"] -= 12                                              # the synthetic pair's disparity: true correspondences
            k2, d2 = f.compute(R, kr, kind)
            m = f.stereo_match(k, d, k2, d2, FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, max_dy=0.7), kind=kind)
            q, t, dist = omatch.stereo_match_crosscheck(k["y"], k2["y"], d, d2, 0.7)
            assert len(q) > 20 and np.array_equal(m["queryIdx"], q) and np.array_equal(m["trainIdx"], t)
            assert np.array_equal(m["distance"], dist)
        with pytest.raises(FE.FeError):
            f.set_brief_pattern(np.full((n_bytes * 8, 4), 25, np.int8))     # offsets outside the 48-px patch


# ---- cv::FREAK (bin/detect_node:43-45; "FREAK" in the descriptor lists of bin/result_ONE:25) -------------------------------
@pytest.mark.parametrize("orient,scale_norm,pscale,octaves", [(True, True, 22.0, 4), (False, True, 22.0, 4), (True, False, 22.0, 4),
                                                              (True, True, 9.0, 3)])
def test_freak_descriptors_vs_oracle(FE, orient, scale_norm, pscale, octaves):
    """FREAK with caller-supplied selected pairs (PARITY UNPINNED: no FREAK binary, OpenCV's default pair table is not in this
    image): kept keypoints, kp.angle bits and all 512 descriptor bits equal the restatement of xfeatures2d/src/freak.cpp
    (pattern table, border rule, integral-image means, integer orientation sums, SSE bit order).  patternScale 9 reaches the
    sigma < 0.5 bilinear branch; mixed keypoint sizes reach several pattern scales."""
    from oracle import freak as ofreak
    L, _ = synth.stereo_pair(240, 320, 33)
    xs, ys, _ = ofast.fast_detect(L, 25, 16, True)
    n = min(len(xs), 500)
    pick = np.linspace(0, len(xs) - 1, n).astype(int)
    kps = np.zeros(n, FE.KPOINT)
    kps["x"], kps["y"] = xs[pick] + np.float32(0.25) * (pick % 4), ys[pick] + np.float32(0.5) * (pick % 2)
    kps["size"] = np.array([7, 7, 9.5, 14, 31, 5], np.float32)[pick % 6]
    sel = ofreak.random_selection(seed=octaves)
    keep, ang, want, _ = ofreak.freak_compute(L, kps["x"], kps["y"], kps["size"], sel, orient, scale_norm, pscale, octaves)
    with FE.FrontEnd(max_width=320, max_height=240, max_keypoints=2048) as f:
        with pytest.raises(FE.FeError):
            f.compute(L, kps, FE.DESC_FREAK)                          # not configured yet
        with pytest.raises(FE.FeError):
            f._check(f.lib.fe_set_freak(f.h, 1, 1, 22.0, 4, None))   # OpenCV's default pair table is not shipped
        f.set_freak(sel, orient, scale_norm, pscale, octaves)
        k, d = f.compute(L, kps, FE.DESC_FREAK)
    assert 0 < keep.sum() < n and len(k) == keep.sum() and d.shape == want.shape
    assert np.array_equal(k["x"], kps["x"][keep]) and np.array_equal(k["size"], kps["size"][keep])
    assert np.array_equal(k["angle"].view(np.uint32), ang.view(np.uint32))
    assert np.array_equal(d, want)
    if orient:
        assert len(np.unique(np.rint(ang / 20))) > 8                 # orientations actually vary


def test_wide_binary_rows_through_the_matchers(FE):
    """64-byte rows (BRIEF-64, FREAK: "BRIEF_64" / "FREAK" of bin/result_ONE:25) through the reference's three matcher call
    sites: knnMatch(q, t, 2, mask) under the epipolar band, the window box and no mask; the Lowe ratio; crossCheck with and
    without the |dy| filter.  Bit-exact against the oracle's BFMatcher restatement (ties -> lowest index: the rows contain
    exact duplicates), ragged counts (not multiples of the 128-row tile), an empty side."""
    from oracle import freak as ofreak
    L, R = synth.stereo_pair(240, 320, 41)
    xs, ys, _ = ofast.fast_detect(L, 25, 16, True)
    pick = np.linspace(0, len(xs) - 1, min(len(xs), 700)).astype(int)
    kl = np.zeros(len(pick), FE.KPOINT)
    kl["x"], kl["y"], kl["size"] = xs[pick], ys[pick], 7
    kr = kl.copy()
    kr["x"] -= 12                                                    # the synthetic pair's disparity
    sel = ofreak.random_selection(seed=1)
    with FE.FrontEnd(max_width=320, max_height=240, max_keypoints=2048) as f:
        f.set_freak(sel)
        kl, dl = f.compute(L, kl, FE.DESC_FREAK)
        kr, dr = f.compute(R, kr, FE.DESC_FREAK)
        assert len(kl) > 300 and len(kr) > 300 and dl.shape[1] == 64
        kr, dr = kr[:-37], dr[:-37].copy()                           # ragged, different counts
        dr[5], dr[9] = dr[200], dr[200]                              # exact duplicates: first minimum wins
        D = omatch.hamming_matrix(dl, dr)
        for cfg, mask in ((FE.match_cfg(mask=FE.MASK_EPIPOLAR, epi_threshold=2.0), omatch.epipolar_mask(kl["y"], kr["y"], 2.0)),
                          (FE.match_cfg(mask=FE.MASK_WINDOW, win_w=100, win_h=60), omatch.window_mask(kl["x"], kl["y"], kr["x"], kr["y"], 100, 60)),
                          (FE.match_cfg(mask=FE.MASK_NONE), None)):
            idx, dist = f.knnMatch(kl, dl, kr, dr, cfg, kind=FE.DESC_FREAK)
            oi, od, _ = omatch.knn2(D, mask)
            assert np.array_equal(idx, oi) and np.array_equal(dist, od)
            m = f.stereo_match(kl, dl, kr, dr, cfg, kind=FE.DESC_BRIEF64)
            q, t, d = omatch.lowe_ratio(oi, od, 0.8)
            assert len(q) > 50 and np.array_equal(m["queryIdx"], q) and np.array_equal(m["trainIdx"], t) and np.array_equal(m["distance"], d)
        for max_dy in (-1.0, 0.7):
            m = f.stereo_match(kl, dl, kr, dr, FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, max_dy=max_dy), kind=FE.DESC_FREAK)
            if max_dy < 0:
                q, t, d = omatch.cross_check(D)
            else:
                q, t, d = omatch.stereo_match_crosscheck(kl["y"], kr["y"], dl, dr, 0.7)
            assert len(q) > 100 and np.array_equal(m["queryIdx"], q) and np.array_equal(m["trainIdx"], t) and np.array_equal(m["distance"], d)
        m = f.window_match(kl, dl, kr, dr, kind=FE.DESC_FREAK)
        q, t, d = omatch.window_match(np.stack([kl["x"], kl["y"]], 1), np.stack([kr["x"], kr["y"]], 1), dl, dr)
        assert np.array_equal(m["queryIdx"], q) and np.array_equal(m["trainIdx"], t)
        assert len(f.stereo_match(kl, dl, kr[:0], dr[:0], FE.match_cfg(mask=FE.MASK_NONE), kind=FE.DESC_FREAK)) == 0
        with pytest.raises(FE.FeError):
            f.stereo_match(kl, dl, kr, dr, FE.match_cfg(mask=FE.MASK_NONE, norm=FE.NORM_HAMMING2), kind=FE.DESC_FREAK)


# ---- the reference's ORB parameter table: edgeThreshold, patchSize, nLevels, scaleFactor, WTA_K combined -----------------
@pytest.mark.parametrize("tag", ["e5p31", "e15p30", "e5p10", "e25p50", "e15p30l2s14w3", "e35p10l4s11w4"])
def test_orb_parameter_table_vs_cv2_golden(FE, tag):
    """cv2.ORB_create(N, scaleFactor, nlevels, edgeThreshold, 0, WTA_K, FAST_SCORE, patchSize, 15).detectAndCompute for
    the parameter ranges of features.py:292-352 (keypoints down to 5 px from the border, intensity-centroid discs and
    rBRIEF patterns of other sizes, 2 / 4 levels at scale 1.4 / 1.1, WTA_K 3 / 4): bit-exact keypoints and descriptors."""
    g = golden("orb_params")
    img = g["img"]
    n, lv, edge, wta, patch = (int(v) for v in g[tag + "_params"])
    with FE.FrontEnd(max_width=img.shape[1], max_height=img.shape[0], max_keypoints=4096, n_features=n, edge_threshold=edge) as f:
        f.setPatchSize(patch)
        f.setWTA_K(wta)
        f.set_pyramid(lv, float(g[tag + "_scale"]))
        k, d, _, _, _ = f.stereo_features(img, img)
    for fld in ("x", "y", "octave", "size", "angle", "response"):
        assert np.array_equal(k[fld], g["%s_%s" % (tag, fld)]), fld
    assert np.array_equal(d, g[tag + "_desc"])


@pytest.mark.gpu
def test_bench_gpu_arm_line_has_the_contract_keys(tmp_path):
    """bench.py's own arm on a small batch: ONE JSON line carrying the contract's keys (metric / value / e2e with real copy
    bytes / roofline / clocks / gpu_launches) and, with FE_BENCH_PHASED=1, both copy schedules.  --dump-outputs writes the
    last timed step's results as float arrays that agree with the line's counts."""
    import json, os, subprocess, sys
    env = dict(os.environ, FE_BENCH_PHASED="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT_DIR, "bench.py"), "--steps", "2", "--warmup", "3", "--pairs", "8", "--no-cpu",
                        "--dump-outputs", str(tmp_path / "dump")],
                       capture_output=True, text=True, timeout=900, cwd=ROOT_DIR, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.strip().splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline", "fabric", "e2e_steady"):
        assert k in d, k
    assert d["value"] > 0 and d["unit"] == "pairs/s" and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 3
    assert d["gpu_launches"] >= 2 * 15 and d["dtype"] == "u8" and d["scaling"] == "weak" and d["vs_baseline"] is None
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 2 * 8 * 1280 * 720 and e["d2h_bytes_per_step"] > 8 * 2 * 5000 * 60
    assert e["value"] < d["value"] * 1.05                       # end to end cannot beat the resident-input rate
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["unit"] in ("GB/s", "TFLOP/s") and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert set(d["e2e_schedules"]) == {"overlapped", "phased"} and e["schedule"] in ("overlapped", "phased")
    assert d["clocks"]["sm_mhz"] > 0 and isinstance(d["clocks"]["reasons"], list)
    dump = {f[:-4]: np.load(tmp_path / "dump" / f) for f in os.listdir(tmp_path / "dump")}
    assert all(v.dtype in (np.float32, np.float64) for v in dump.values())
    assert dump["n_kps"].mean() == d["counts"]["keypoints_per_image_mean"] and dump["n_a"].mean() == d["counts"]["ratio_matches_per_pair_mean"]
    assert dump["n_b"].mean() == d["counts"]["crosscheck_matches_per_pair_mean"] and dump["pairs"].tolist() == list(range(8))
    for e in range(16):
        m = int(dump["n_kps"][e])
        k = dump["kps"][e // 2, e % 2]
        assert m > 1000 and np.all((k[:m, 0] > 0) & (k[:m, 0] < 1280) & (k[:m, 1] > 0) & (k[:m, 1] < 720)) and not k[m:].any()
