"""BRIEF-16 / BRIEF-32 in the batched stereo pipeline and fe_stereo_features (BRIEF-64 there too).

The batch's semantics are detector.detect followed by BriefDescriptorExtractor::compute: the detector's keypoints (top-N
or Harris cut first), then runByImageBorder(28), then the tests.  Every comparison with a device entry point is bit for bit:
keypoint records, descriptor bytes, match indices and distance bits.  The oracle (oracle/brief.py, oracle/match.py) is
integer-exact as well, so it is compared bit for bit too.  The test tables are seeded random stand-ins for OpenCV's.
"""
import numpy as np
import pytest

from oracle import brief as obrief
from oracle import match as omatch
from oracle import synth
from test_join128_scenario import band_candidates, join128_scenario

pytestmark = pytest.mark.gpu

H, W = 360, 480          # neither a multiple of the 64-row nor of the 256-column tile


@pytest.fixture(scope="module")
def FE(fe):
    return fe


def _tables():
    return {16: obrief.random_tests(16, 7), 32: obrief.random_tests(32, 8), 64: obrief.random_tests(64, 9)}


def _kind(FE, n_bytes):
    return {16: FE.DESC_BRIEF16, 32: FE.DESC_BRIEF32, 64: FE.DESC_BRIEF64}[n_bytes]


def _same_bits(a, b):
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def _pairs(P, h=H, w=W, seed=0):
    ps = [synth.stereo_pair(h, w, seed + p) for p in range(P)]
    return np.stack([p[0] for p in ps]), np.stack([p[1] for p in ps])


DETECTORS = {
    "orb": dict(n_features=1500, edge_threshold=31, orientation=True),
    "fastx": dict(n_features=-1, edge_threshold=0, orientation=False, fast_threshold=20),
}


def _front(FE, P, h=H, w=W, cap=16384, **det):
    return FE.FrontEnd(max_width=w, max_height=h, max_pairs=P, max_keypoints=cap, **det)


def _brief_ctx(FE, f, n_bytes, orient=False):
    tabs = _tables()
    f.set_brief_pattern(tabs[n_bytes], use_orientation=orient)
    f.set_batch_descriptor(_kind(FE, n_bytes))
    return tabs[n_bytes]


def _batch(f, Ls, Rs, cfg_a=None, cfg_b=None):
    f.batch_upload(Ls, Rs)
    f.batch_run(cfg_a, cfg_b, sync=True)
    return f.batch_download()


def _image(out, i):
    n = out["n_kps"][i]
    return out["kps"][i][:n], out["desc"][i][:n]


def _bordered(k, h, w):
    return k[obrief.keep_mask(k["x"], k["y"], w, h)]


def _check_image(FE, f, img, k, d, tab, n_bytes, orient):
    """The batch's keypoints are the detector's minus the 28-px band, its rows those of fe_describe and of the oracle."""
    h, w = img.shape
    assert _same_bits(k, _bordered(f.detect(img), h, w))
    assert d.shape == (len(k), n_bytes)
    kk, dd = f.compute(img, k, _kind(FE, n_bytes))
    assert _same_bits(kk, k) and _same_bits(dd, d)
    keep, want = obrief.brief_compute(img, k["x"], k["y"], tab, k["angle"], orient)
    assert keep.all() and _same_bits(want, d)


def _cfg_a(FE):
    return FE.match_cfg()                                                    # |dy| <= 2, Lowe 0.8


def _cfg_b(FE):
    return FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, max_dy=0.7)


# ---- 1. rows -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("det", sorted(DETECTORS))
@pytest.mark.parametrize("orient", [False, True])
@pytest.mark.parametrize("n_bytes", [16, 32])
def test_batch_rows_equal_describe_and_oracle(FE, n_bytes, orient, det):
    Ls, Rs = _pairs(2, seed=3)
    with _front(FE, 2, **DETECTORS[det]) as f:
        tab = _brief_ctx(FE, f, n_bytes, orient)
        out = _batch(f, Ls, Rs)
        for i in range(4):
            img = (Ls, Rs)[i & 1][i >> 1]
            k, d = _image(out, i)
            assert len(k) > 300, (i, len(k))
            assert np.all(np.diff(k["y"]) >= 0)                          # raster order survives the compaction
            _check_image(FE, f, img, k, d, tab, n_bytes, orient)


# ---- 2. the border after the top-N / Harris cut --------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ["fast_score", "harris", "pyramid"])
def test_border_applies_after_the_detector(FE, variant):
    """edge_threshold 5 with a small n_features: some of the top N lie inside the 28-px band.  The batch keeps the detector's
    keypoints outside the band (detect, then filter), which differs from filtering first and taking the top N then."""
    Ls, Rs = _pairs(1, seed=11)
    n, tab = 300, _tables()[32]
    with _front(FE, 1, n_features=n, edge_threshold=5) as f, _front(FE, 1, n_features=n, edge_threshold=28) as g:
        for ctx in (f, g):
            if variant == "harris":
                ctx.setScoreType(0)
            if variant == "pyramid":
                ctx.set_pyramid(3, 1.2)
        _brief_ctx(FE, f, 32, orient=True)
        out = _batch(f, Ls, Rs)
        for i, img in enumerate((Ls[0], Rs[0])):
            k, d = _image(out, i)
            det = f.detect(img)
            in_band = len(det) - len(_bordered(det, H, W))
            assert in_band > 0, (variant, i)
            filter_first = g.detect(img)                                 # runByImageBorder(28), then the top N
            assert not _same_bits(k, filter_first), (variant, i)
            _check_image(FE, f, img, k, d, tab, 32, True)


# ---- 3. tile edges -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hw", [(200, 300), (130, 530), (64, 257), (71, 600)])
def test_tile_edges_and_odd_sizes(FE, hw):
    """Sizes that are not multiples of 16, 64 or 256, with dense FAST keypoints on tile rows 63 / 64, columns 255 / 256 and
    the last kept row / column (h - 29, w - 29)."""
    h, w = hw
    Ls, Rs = _pairs(1, h, w, seed=h + w)
    tab = _tables()[16]
    with _front(FE, 1, h, w, fast_threshold=8, n_features=-1, edge_threshold=0, orientation=False) as f:
        _brief_ctx(FE, f, 16, orient=True)
        out = _batch(f, Ls, Rs)
        ks = []
        for i, img in enumerate((Ls[0], Rs[0])):
            k, d = _image(out, i)
            _check_image(FE, f, img, k, d, tab, 16, True)
            ks.append(k)
        x, y = np.concatenate([k["x"] for k in ks]), np.concatenate([k["y"] for k in ks])
        assert np.any(y == h - 29) and np.any(x == w - 29)
        if h > 92:
            assert np.any(y == 63) and np.any(y == 64)
        if w > 284:
            assert np.any(x == 255) and np.any(x == 256)


def test_truncated_boxes_at_the_border(FE):
    """Keypoints whose coordinates round up onto the border ((int)(y + 0.5) = h - 28, x likewise) under tests at offset
    +24: the boxes reach one row / column past the image (brief_kernel clamps the integral-image index).  Checked through
    fe_describe only.  Integer detector keypoints end at h - 29, so brief_tile_kernel never meets such boxes; a pyramid
    batch can (its fractional keypoints go through brief_kernel), but no test here plants one there."""
    h, w = 150, 170
    img = synth.stereo_pair(h, w, 5)[0]
    tab = _tables()[32].copy()
    tab[:64] = (24, 24, -24, -24)
    tab[64:128] = (24, -3, 0, 24)
    with _front(FE, 1, h, w) as f:
        f.set_brief_pattern(tab)
        k = np.zeros(4, FE.KPOINT)
        k["x"] = (w - 28.4, 60.0, w - 28.01, 28.0)
        k["y"] = (h - 28.3, h - 28.45, 80.0, 28.0)
        k["size"] = 31
        kk, d = f.compute(img, k, FE.DESC_BRIEF32)
        keep, want = obrief.brief_compute(img, k["x"], k["y"], tab)
        assert keep.all() and _same_bits(kk, k) and _same_bits(d, want)


def test_empty_side_and_tiny_images(FE):
    """One side without keypoints (a flat image) matches nothing; an image under 57 px keeps no keypoint."""
    Ls, Rs = _pairs(2, seed=21)
    Rs[1][:] = 128
    with _front(FE, 2, **DETECTORS["orb"]) as f:
        tab = _brief_ctx(FE, f, 32)
        out = _batch(f, Ls, Rs, _cfg_a(FE), _cfg_b(FE))
        assert out["n_kps"][3] == 0 and out["n_a"][1] == 0 and out["n_b"][1] == 0
        k, d = _image(out, 2)
        _check_image(FE, f, Ls[1], k, d, tab, 32, False)
        assert out["n_a"][0] > 100 and out["n_b"][0] > 100
    Ls, Rs = _pairs(1, 56, 80, seed=2)
    with _front(FE, 1, 56, 80, fast_threshold=5, n_features=-1, edge_threshold=0, orientation=False) as f:
        _brief_ctx(FE, f, 16)
        assert len(f.detect(Ls[0])) > 0
        out = _batch(f, Ls, Rs, _cfg_a(FE), _cfg_b(FE))
        assert list(out["n_kps"]) == [0, 0] and out["n_a"][0] == 0 and out["n_b"][0] == 0


# ---- 4. matching ---------------------------------------------------------------------------------------------------------
def _check_matches(FE, f, out, P, n_bytes):
    kind = _kind(FE, n_bytes)
    for p in range(P):
        lk, ld = _image(out, 2 * p)
        rk, rd = _image(out, 2 * p + 1)
        ma = out["matches_a"][p][:out["n_a"][p]]
        mb = out["matches_b"][p][:out["n_b"][p]]
        assert len(ma) > 50 and len(mb) > 50, (p, len(ma), len(mb))
        assert _same_bits(f.stereo_match(lk, ld, rk, rd, _cfg_a(FE), kind), ma), p
        assert _same_bits(f.stereo_match(lk, ld, rk, rd, _cfg_b(FE), kind), mb), p
        for m, (q, t, d) in ((ma, omatch.stereo_match_ratio(lk["y"], rk["y"], ld, rd, 2.0, 0.8)),
                             (mb, omatch.stereo_match_crosscheck(lk["y"], rk["y"], ld, rd, 0.7))):
            assert np.array_equal(m["queryIdx"], q) and np.array_equal(m["trainIdx"], t)
            assert np.array_equal(m["distance"], d.astype(np.float32))


@pytest.mark.parametrize("n_bytes", [16, 32])
def test_batch_matching_equals_host_and_oracle(FE, n_bytes):
    P = 3
    Ls, Rs = _pairs(P, seed=31)
    with _front(FE, P, **DETECTORS["orb"]) as f:
        _brief_ctx(FE, f, n_bytes, orient=True)
        out = _batch(f, Ls, Rs, _cfg_a(FE), _cfg_b(FE))
        _check_matches(FE, f, out, P, n_bytes)


# ---- 5. the multi-index join on 128-bit rows -----------------------------------------------------------------------------
@pytest.mark.parametrize("n", [0, 1, 257, 4097])
def test_cross_check_join_on_128_bit_rows(FE, n):
    """join128_scenario (tests/test_join128_scenario.py): band pairs at 7 and 8 bits that lose their row or column to class-A
    entries outside the band -- ties at a lower index and closer partners, with one identical data half at 7 bits and none
    at 8 -- and ties at a higher index that do not.  A class-A bound of 8, or a join that finds nothing, fails here."""
    qd, qy, td, ty = join128_scenario(n, n, n + 3)
    qk, tk = np.zeros(len(qy), FE.KPOINT), np.zeros(len(ty), FE.KPOINT)
    qk["y"], tk["y"] = qy, ty
    with _front(FE, 1, 64, 64) as f:
        f.profile_reset()
        got = f.stereo_match(qk, qd, tk, td, _cfg_b(FE), FE.DESC_BRIEF16)
        assert f.stage_times()["hamming_cross"][1] == 11                  # the pruned path with the join ran
    q, t, d = omatch.stereo_match_crosscheck(qy, ty, qd, td, 0.7)
    assert np.array_equal(got["queryIdx"], q) and np.array_equal(got["trainIdx"], t)
    assert np.array_equal(got["distance"], d.astype(np.float32))
    if n > 1:
        assert len(q) > n // 8 and set(np.unique(d)) >= {7, 8}
        cands, _, _ = band_candidates(omatch.hamming_matrix(qd, td).astype(np.int64), qy, ty)
        kept = set(zip(q.tolist(), t.tolist()))
        killed = {dd for i, j, dd in cands if dd <= 8 and (i, j) not in kept}
        assert killed == {7, 8}                                           # out-of-band disturbers at both class edges


# ---- 6. landmarks and the window -----------------------------------------------------------------------------------------
def _sequence(F, seed):
    fr = synth.stereo_sequence(H, W, seed, F)
    return np.stack([p[0] for p in fr]), np.stack([p[1] for p in fr])


def _landmarks(out, fr, which="a"):
    m = out["matches_" + which][fr][:out["n_" + which][fr]]
    return (out["kps"][2 * fr][m["queryIdx"]], out["desc"][2 * fr][m["queryIdx"]],
            out["kps"][2 * fr + 1][m["trainIdx"]], out["desc"][2 * fr + 1][m["trainIdx"]], m)


@pytest.mark.parametrize("n_bytes", [16, 32])
def test_landmarks_and_window(FE, n_bytes):
    F = 4
    Ls, Rs = _sequence(F, 41)
    kind = _kind(FE, n_bytes)
    live = FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE)
    cc = FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, max_dy=-1.0)
    with _front(FE, F, **DETECTORS["orb"]) as f:
        _brief_ctx(FE, f, n_bytes, orient=True)
        out = _batch(f, Ls, Rs, _cfg_a(FE), _cfg_b(FE))
        for which in (0, 1):
            pk = f.batch_landmarks(which)
            assert pk["l_desc"].dtype == np.uint8 and pk["l_desc"].shape[2] == n_bytes
            for fr in range(F):
                lk, ld, rk, rd, m = _landmarks(out, fr, "ab"[which])
                n = len(m)
                assert pk["n"][fr] == n and n > 50
                assert _same_bits(pk["l_kps"][fr][:n], lk) and _same_bits(pk["r_kps"][fr][:n], rk)
                assert _same_bits(pk["l_desc"][fr][:n], ld) and _same_bits(pk["r_desc"][fr][:n], rd)
                assert _same_bits(pk["matches"][fr][:n]["distance"], m["distance"])
        tracks, n_tr, _ = f.window_batch()
        live_tracks, n_live, _ = f.window_batch(cfg=live)
        lm = [_landmarks(out, fr) for fr in range(F)]
        for fr in range(1, F):
            cur, prev = lm[fr], lm[fr - 1]
            got = tracks[fr - 1][:n_tr[fr - 1]]
            assert len(got) > 50
            assert _same_bits(f.window_match(cur[0], cur[1], prev[0], prev[1], kind=kind), got), fr
            ml = f.stereo_match(cur[0], cur[1], prev[0], prev[1], cc, kind)
            mr = f.stereo_match(cur[2], cur[3], prev[2], prev[3], cc, kind)
            right = dict(zip(mr["queryIdx"].tolist(), mr["trainIdx"].tolist()))
            keep = np.array([right.get(a, -1) == b for a, b in zip(ml["queryIdx"].tolist(), ml["trainIdx"].tolist())], bool)
            assert _same_bits(live_tracks[fr - 1][:n_live[fr - 1]], ml[keep]), fr
        f.window_update(reset=True)
        for fr in range(F):
            got, frames = f.window_update(lm[fr][0], lm[fr][1], cfg=FE.match_cfg(mask=FE.MASK_WINDOW), kind=kind)
            if fr:
                assert _same_bits(got, tracks[fr - 1][:n_tr[fr - 1]]), fr


# ---- 7. the overlapped pipeline ------------------------------------------------------------------------------------------
def test_pipeline_chunks_equal_upload_run_download(FE):
    P = 5
    Ls, Rs = _pairs(P, seed=51)
    with _front(FE, P, **DETECTORS["orb"]) as f:
        _brief_ctx(FE, f, 16, orient=True)
        f.set_chunk_pairs(2)
        piped = f.pipeline_batch(Ls, Rs, _cfg_a(FE), _cfg_b(FE))
        ref = _batch(f, Ls, Rs, _cfg_a(FE), _cfg_b(FE))
    for i in range(2 * P):
        assert _same_bits(_image(piped, i)[0], _image(ref, i)[0]) and _same_bits(_image(piped, i)[1], _image(ref, i)[1])
    for p in range(P):
        for w in "ab":
            n = ref["n_" + w][p]
            assert piped["n_" + w][p] == n and n > 50
            assert _same_bits(piped["matches_" + w][p][:n], ref["matches_" + w][p][:n])


# ---- 8. switching descriptors --------------------------------------------------------------------------------------------
def test_switching_descriptors_keeps_orb(FE):
    P = 2
    Ls, Rs = _pairs(P, seed=61)
    with _front(FE, P, **DETECTORS["orb"]) as fresh:
        want = _batch(fresh, Ls, Rs, _cfg_a(FE), _cfg_b(FE))
    with _front(FE, P, **DETECTORS["orb"]) as f:
        _batch(f, Ls, Rs, _cfg_a(FE), _cfg_b(FE))
        _brief_ctx(FE, f, 32)
        _batch(f, Ls, Rs, _cfg_a(FE), _cfg_b(FE))
        f.set_batch_descriptor(FE.DESC_ORB256)
        got = _batch(f, Ls, Rs, _cfg_a(FE), _cfg_b(FE))
    for key in ("n_kps", "n_a", "n_b"):
        assert np.array_equal(got[key], want[key]), key
    for i in range(2 * P):
        assert _same_bits(_image(got, i)[0], _image(want, i)[0]) and _same_bits(_image(got, i)[1], _image(want, i)[1]), i
    for p in range(P):                  # (rows past a pair's count are not written: the slabs hold what earlier runs left)
        for w in "ab":
            n = want["n_" + w][p]
            assert _same_bits(got["matches_" + w][p][:n], want["matches_" + w][p][:n]), (p, w)


# ---- 9. fe_stereo_features -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_bytes", [16, 32, 64])
def test_stereo_features_brief(FE, n_bytes):
    L, R = synth.stereo_pair(H, W, 71)
    with _front(FE, 1, **DETECTORS["orb"]) as f:
        tab = _tables()[n_bytes]
        f.set_brief_pattern(tab, use_orientation=n_bytes != 32)
        lk, ld, rk, rd, _ = f.stereo_features(L, R, kind=_kind(FE, n_bytes))
        for img, k, d in ((L, lk, ld), (R, rk, rd)):
            assert len(k) > 300
            _check_image(FE, f, img, k, d, tab, n_bytes, n_bytes != 32)


# ---- 10. errors ----------------------------------------------------------------------------------------------------------
def _code(FE, fn, *args, **kw):
    with pytest.raises(FE.FeError) as e:
        fn(*args, **kw)
    return e.value.code


def test_unsupported_configurations(FE):
    U = FE.lib.FE_ERR_UNSUPPORTED
    Ls, Rs = _pairs(1, seed=81)
    with _front(FE, 1) as f:
        assert _code(FE, f.set_batch_descriptor, FE.DESC_BRIEF16) == U                # no table
        f.set_brief_pattern(_tables()[64])
        assert _code(FE, f.set_batch_descriptor, FE.DESC_BRIEF32) == U                # only a table of another width
        assert _code(FE, f.set_batch_descriptor, FE.DESC_BRIEF64) == U                # 512-bit rows
        assert _code(FE, f.set_batch_descriptor, FE.DESC_FREAK) == U
        f.set_brief_pattern(_tables()[32])
        f.set_batch_descriptor(FE.DESC_BRIEF32)
        f.batch_upload(Ls, Rs)
        for cfg in (FE.match_cfg(norm=FE.NORM_L2), FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, norm=FE.NORM_L2)):
            assert _code(FE, f.batch_run, cfg, None, sync=True) == U
        f.set_batch_detector({})
        assert _code(FE, f.set_batch_descriptor, FE.DESC_BRIEF32) == U                # a Fast-Hessian ctx
    with _front(FE, 1) as f:
        assert _code(FE, f.stereo_features, Ls[0], Rs[0], kind=FE.DESC_BRIEF16) == U


# ---- 11. full size -------------------------------------------------------------------------------------------------------
def test_full_size(FE):
    P = 4
    Ls, Rs = _pairs(P, 720, 1280, seed=91)
    with _front(FE, P, 720, 1280, cap=16384, n_features=5000) as f:
        _brief_ctx(FE, f, 32, orient=True)
        out = _batch(f, Ls, Rs, _cfg_a(FE), _cfg_b(FE))
        assert np.all(out["n_kps"] > 3000)
        _check_matches(FE, f, out, P, 32)
