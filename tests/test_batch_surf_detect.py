"""The batched pipeline with SURF's Fast-Hessian detector (fe_set_batch_detector): the service chain
getStereoFeatures(SURF, SURF) -> stereoMatching -> windowMatching on the device.

The batch's keypoints are the survivors of fe_surf_detect_batch in raster order (y, x, then KeypointGreater), so every
image is demanded bit for bit equal to the single-entry detector's output re-sorted on the host; its matches, landmarks
and tracks bit for bit equal to the host entry points (fe_stereo_match, fe_window_match) on the batch's own downloaded
keypoints and rows, and within the north-star tolerance of the numpy matcher (>= 99.9 % agreement; the oracle's L2 is
evaluated in float64, not in the device's FP32 order).
"""
import numpy as np
import pytest

from oracle import match as omatch
from oracle import synth

pytestmark = pytest.mark.gpu

H, W = 360, 480
# (hessian_threshold, n_octaves, n_octave_layers, oriented / upright, SURF-64 / SURF-128); n_octaves = 1 keeps every window
# (at most 21 * 27 * 1.2 / 9 = 75 px) inside the staged describe kernel
PARAMS = [dict(hessian_threshold=100.0, n_octaves=4, n_octave_layers=2, upright=False, extended=False),
          dict(hessian_threshold=150.0, n_octaves=3, n_octave_layers=2, upright=True, extended=True),
          dict(hessian_threshold=100.0, n_octaves=1, n_octave_layers=2, upright=False, extended=True)]
PARAM_IDS = ["t100-o4-oriented-64", "t150-o3-upright-128", "t100-o1-oriented-128"]


@pytest.fixture(scope="module")
def FE(fe):
    return fe


def _kind(FE, surf):
    return FE.DESC_SURF128 if surf.get("extended") else FE.DESC_SURF64


def _cfg_a(FE):
    return FE.match_cfg(norm=FE.NORM_L2)                                   # |dy| <= 2, Lowe 0.8


def _cfg_b(FE):
    return FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, norm=FE.NORM_L2, max_dy=0.7)


def _same_bits(a, b):
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def _interleave(Ls, Rs):
    """Images in the batch's slot order: left of pair p at 2p, right at 2p + 1."""
    return np.stack([im for p in range(len(Ls)) for im in (Ls[p], Rs[p])])


def _raster(kps, desc):
    """The single-entry output (KeypointGreater order) in the batch's order: y, then x, then KeypointGreater."""
    o = np.lexsort((np.arange(len(kps)), kps["x"], kps["y"]))
    return kps[o], desc[o]


def _batch(f, Ls, Rs, cfg_a=None, cfg_b=None):
    f.batch_upload(Ls, Rs)
    f.batch_run(cfg_a, cfg_b, sync=True)
    return f.batch_download()


def _image(out, i):
    n = out["n_kps"][i]
    return out["kps"][i][:n], out["desc"][i][:n]


def _check_against_single_entry(f, surf, Ls, Rs, out):
    kps, desc = f.surf_detect_batch(_interleave(Ls, Rs), **surf)
    for i in range(2 * len(Ls)):
        k, d = _image(out, i)
        want_k, want_d = _raster(kps[i], desc[i])
        assert len(k) > 100 and len(k) == len(want_k), (i, len(k), len(want_k))
        assert np.all(k["size"] > 0) and np.all(np.diff(k["y"]) >= 0), i
        assert _same_bits(k, want_k), i
        assert _same_bits(d, want_d), i


class Agreement:
    """Oracle matches the device reproduces (same query, same train; distance within rtol 1e-5), summed over pairs."""

    def __init__(self):
        self.want = self.hit = self.got = 0

    def add(self, got, q, t, d):
        g = {int(a): (int(b), float(c)) for a, b, c in zip(got["queryIdx"], got["trainIdx"], got["distance"])}
        for qi, ti, di in zip(q.tolist(), t.tolist(), d.tolist()):
            m = g.get(qi)
            if m is not None and m[0] == ti:
                assert np.isclose(m[1], di, rtol=1e-5, atol=0), (qi, ti, m[1], di)
                self.hit += 1
        self.want += len(q)
        self.got += len(got)

    def check(self):
        assert self.want > 0 and self.hit >= 0.999 * self.want, (self.hit, self.want)
        assert self.got <= 1.001 * self.want + 1, (self.got, self.want)


def _check_matches(FE, f, surf, out, pairs, oracle_pairs):
    """Mode A and mode B of the batch against fe_stereo_match on the batch's own keypoints and rows (bit for bit) and
    against the numpy matcher (>= 99.9 %)."""
    kind = _kind(FE, surf)
    cc = FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, norm=FE.NORM_L2, max_dy=0.7)
    agree_a, agree_b = Agreement(), Agreement()
    for p in range(pairs):
        lk, ld = _image(out, 2 * p)
        rk, rd = _image(out, 2 * p + 1)
        lk, ld, rk, rd = (np.ascontiguousarray(a) for a in (lk, ld, rk, rd))
        ma = out["matches_a"][p][:out["n_a"][p]]
        mb = out["matches_b"][p][:out["n_b"][p]]
        assert len(ma) > 50 and len(mb) > 50, (p, len(ma), len(mb))
        assert _same_bits(ma, f.stereo_match(lk, ld, rk, rd, _cfg_a(FE), kind=kind)), p
        assert _same_bits(mb, f.stereo_match(lk, ld, rk, rd, cc, kind=kind)), p
        if p < oracle_pairs:
            agree_a.add(ma, *omatch.stereo_match_ratio(lk["y"], rk["y"], ld, rd, 2.0, 0.8, norm="l2"))
            agree_b.add(mb, *omatch.stereo_match_crosscheck(lk["y"], rk["y"], ld, rd, 0.7, norm="l2"))
    agree_a.check()
    agree_b.check()


@pytest.mark.parametrize("surf", PARAMS, ids=PARAM_IDS)
def test_batch_equals_single_entry_detector(FE, surf):
    """Both eyes of three pairs: every fe_kpoint field and every descriptor float of the batch equal fe_surf_detect_batch's
    output in raster order; no record of size <= 0, y non-decreasing."""
    P = 3
    Ls, Rs = synth.stereo_batch(H, W, P, seed0=11)
    with FE.FrontEnd(max_width=W, max_height=H, max_pairs=P, max_keypoints=8192) as f:
        f.set_batch_detector(surf)
        out = _batch(f, Ls, Rs, _cfg_a(FE), _cfg_b(FE))
        _check_against_single_entry(f, surf, Ls, Rs, out)


def _with_discs(img, radii, centres):
    """img with dark discs: blobs whose Hessian maxima lie at box-filter sizes of about 5.3 x the radius."""
    yy, xx = np.mgrid[:img.shape[0], :img.shape[1]]
    out = img.astype(np.int16)
    for r, (cy, cx) in zip(radii, centres):
        out[(yy - cy) ** 2 + (xx - cx) ** 2 <= r * r] -= 90
    return np.clip(out, 0, 255).astype(np.uint8)


def test_batch_drops_what_surf_drops(FE):
    """5 octaves of 4 layers on 1280x720 with dark discs of radius 90-110 px: some of their maxima lie at sizes above 365, whose
    descriptor window exceeds 1024 px, so SURFInvoker drops them.  The batch holds exactly fe_surf_detect_batch's survivors
    and no size <= 0 record; a ctx too small for the maxima reports how many there were, which is more than the survivors."""
    h, w = 720, 1280
    surf = dict(hessian_threshold=100.0, n_octaves=5, n_octave_layers=4, upright=False, extended=False)
    Ls, Rs = synth.stereo_batch(h, w, 1, seed0=5)
    radii, centres = (90, 100, 110), ((360, 300), (360, 640), (360, 980))
    Ls = np.stack([_with_discs(Ls[0], radii, centres)])
    Rs = np.stack([_with_discs(Rs[0], radii, [(cy, cx - 12) for cy, cx in centres])])
    with FE.FrontEnd(max_width=w, max_height=h, max_pairs=1, max_keypoints=64) as f:
        f.set_batch_detector(surf)
        f.batch_upload(Ls, Rs)
        f.batch_run(None, None)
        st, out = _raw_download(f, 1)
        assert st == FE.lib.FE_ERR_CAPACITY
        maxima = out["n_kps"].copy()
    with FE.FrontEnd(max_width=w, max_height=h, max_pairs=1) as f:
        f.set_batch_detector(surf)
        out = _batch(f, Ls, Rs)
        _check_against_single_entry(f, surf, Ls, Rs, out)
        survivors = out["n_kps"].copy()
        assert out["kps"][0][:survivors[0]]["size"].max() <= 365.0
    print("maxima", maxima.tolist(), "survivors", survivors.tolist())
    assert np.all(maxima > survivors), (maxima, survivors)


@pytest.mark.parametrize("surf", PARAMS[:2], ids=PARAM_IDS[:2])
def test_batch_matches_equal_host_matchers(FE, surf):
    """Mode A (|dy| <= 2, Lowe 0.8: the banded L2 kernel) and mode B (cross-check + |dy| <= 0.7: the exact tensor-core
    verification) of fe_batch_run equal fe_stereo_match on the downloaded keypoints and rows bit for bit, and the numpy
    matcher on >= 99.9 % of its matches."""
    P = 3
    Ls, Rs = synth.stereo_batch(H, W, P, seed0=23)
    with FE.FrontEnd(max_width=W, max_height=H, max_pairs=P, max_keypoints=8192) as f:
        f.set_batch_detector(surf)
        out = _batch(f, Ls, Rs, _cfg_a(FE), _cfg_b(FE))
        out = {k: v.copy() for k, v in out.items()}
        _check_matches(FE, f, surf, out, P, P)


def _host_live(FE, f, kind, cur, prev):
    """liveGraph on the host entry point: fe_stereo_match cross-checks of the left rows and of the right rows (no mask, no
    |dy| filter), intersected on the same previous landmark."""
    cc = FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, norm=FE.NORM_L2, max_dy=-1.0)
    ml = f.stereo_match(cur[0], cur[1], prev[0], prev[1], cc, kind=kind)
    mr = f.stereo_match(cur[2], cur[3], prev[2], prev[3], cc, kind=kind)
    right = dict(zip(mr["queryIdx"].tolist(), mr["trainIdx"].tolist()))
    keep = np.array([right.get(q, -1) == t for q, t in zip(ml["queryIdx"].tolist(), ml["trainIdx"].tolist())], bool)
    return ml[keep]


def _landmarks(out, fr, which):
    m = out["matches_a" if which == 0 else "matches_b"][fr][:out["n_a" if which == 0 else "n_b"][fr]]
    return (out["kps"][2 * fr][m["queryIdx"]], out["desc"][2 * fr][m["queryIdx"]],
            out["kps"][2 * fr + 1][m["trainIdx"]], out["desc"][2 * fr + 1][m["trainIdx"]], m)


@pytest.mark.parametrize("surf", PARAMS[:2], ids=PARAM_IDS[:2])
def test_batch_landmarks_and_window_tracks(FE, surf):
    """A 6-frame sequence through fe_pipeline_batch with the Fast-Hessian detector: fe_batch_landmarks (both `which`)
    packs the downloaded matches' keypoints and rows; fe_window_batch in WindowMatcher mode equals fe_window_match and in
    liveGraph mode two fe_stereo_match cross-checks, on the downloaded landmarks."""
    F = 6
    fr_ = synth.stereo_sequence(H, W, 31, F)
    Ls, Rs = np.stack([p[0] for p in fr_]), np.stack([p[1] for p in fr_])
    kind = _kind(FE, surf)
    with FE.FrontEnd(max_width=W, max_height=H, max_pairs=F, max_keypoints=8192) as f:
        f.set_batch_detector(surf)
        out = f.pipeline_batch(Ls, Rs, _cfg_a(FE), _cfg_b(FE))
        out = {k: v.copy() for k, v in out.items()}
        tr_w, n_w, _ = f.window_batch(cfg=FE.match_cfg(mask=FE.MASK_WINDOW, norm=FE.NORM_L2))
        tr_w, n_w = tr_w.copy(), n_w.copy()
        tr_l, n_l, _ = f.window_batch(cfg=FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, norm=FE.NORM_L2))
        tr_l, n_l = tr_l.copy(), n_l.copy()
        packs = [f.batch_landmarks(which) for which in (0, 1)]
        # (host entry points from here on: they reuse the ctx's device slots)
        for which, pk in enumerate(packs):
            assert pk["l_desc"].dtype == np.float32 and pk["l_desc"].shape[2] == (128 if surf["extended"] else 64)
            for fr in range(F):
                lk, ld, rk, rd, m = _landmarks(out, fr, which)
                n = len(m)
                assert n > 20 and pk["n"][fr] == n, (which, fr)
                assert _same_bits(pk["l_kps"][fr][:n], lk) and _same_bits(pk["r_kps"][fr][:n], rk), (which, fr)
                assert _same_bits(pk["l_desc"][fr][:n], ld) and _same_bits(pk["r_desc"][fr][:n], rd), (which, fr)
                assert _same_bits(pk["matches"][fr][:n]["distance"], m["distance"]), (which, fr)
        lm = [tuple(np.ascontiguousarray(a) for a in _landmarks(out, fr, 0)[:4]) for fr in range(F)]
        for fr in range(1, F):
            cur, prev = lm[fr], lm[fr - 1]
            got = tr_w[fr - 1][:n_w[fr - 1]]
            assert len(got) > 20
            one = f.window_match(cur[0], cur[1], prev[0], prev[1], cfg=FE.match_cfg(mask=FE.MASK_WINDOW, norm=FE.NORM_L2),
                                 kind=kind)
            assert _same_bits(one, got), fr
            got = tr_l[fr - 1][:n_l[fr - 1]]
            assert len(got) > 20
            assert _same_bits(got, _host_live(FE, f, kind, cur, prev)), fr


def test_pipeline_batch_two_chunks_equals_upload_run_download(FE):
    """96 pairs: two default chunks, which would take the overlapped two-lane path of fe_pipeline_batch if the Fast-Hessian
    batch did not stay on the single stream (the lanes would share one scale space).  Bit for bit upload / run / download."""
    h, w, P = 120, 160, 96
    surf = dict(hessian_threshold=100.0, n_octaves=3, n_octave_layers=2, upright=False, extended=True)
    Ls, Rs = synth.stereo_batch(h, w, P, seed0=3)
    with FE.FrontEnd(max_width=w, max_height=h, max_pairs=P, max_keypoints=1024) as f:
        f.set_batch_detector(surf)
        a = f.pipeline_batch(Ls, Rs, _cfg_a(FE), _cfg_b(FE))
        a = {k: v.copy() for k, v in a.items()}
        b = _batch(f, Ls, Rs, _cfg_a(FE), _cfg_b(FE))
    assert a["n_kps"].min() > 10 and a["n_a"].sum() > 100 and a["n_b"].sum() > 100
    for k in a:
        assert _same_bits(a[k], b[k]), k


def test_switching_detectors(FE):
    """ORB run -> Fast-Hessian run -> back to FAST with the ORB descriptor: the last run equals the first byte for byte.
    While the Fast-Hessian detector is selected, fe_set_batch_descriptor and Hamming norms are FE_ERR_UNSUPPORTED."""
    P = 2
    Ls, Rs = synth.stereo_batch(H, W, P, seed0=17)
    cc_h = FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE)
    with FE.FrontEnd(max_width=W, max_height=H, max_pairs=P, max_keypoints=8192) as f:
        first = {k: v.copy() for k, v in _batch(f, Ls, Rs, FE.match_cfg(), cc_h).items()}
        f.set_batch_detector({})
        hes = _batch(f, Ls, Rs, _cfg_a(FE), _cfg_b(FE))
        assert hes["desc"].dtype == np.float32 and hes["desc"].shape[2] == 64 and hes["n_kps"].min() > 100
        for call in (lambda: f.set_batch_descriptor(FE.DESC_ORB256), lambda: f.batch_run(FE.match_cfg(), None, sync=True),
                     lambda: f.batch_run(None, cc_h, sync=True)):
            with pytest.raises(FE.FeError) as e:
                call()
            assert e.value.code == FE.lib.FE_ERR_UNSUPPORTED
        f.set_batch_detector(None)
        f.set_batch_descriptor(FE.DESC_ORB256)
        last = _batch(f, Ls, Rs, FE.match_cfg(), cc_h)
        assert last["desc"].dtype == np.uint8
        for k in first:
            assert _same_bits(first[k], last[k]), k


def _raw_download(f, P):
    """fe_batch_download without raising: (status, outputs)."""
    from front_end_b200.frontend import _ptr
    out = f.alloc_batch_outputs(P)
    st = f.lib.fe_batch_download(f.h, f.max_keypoints, _ptr(out["kps"]), _ptr(out["desc"]), _ptr(out["n_kps"]),
                                 _ptr(out["matches_a"]), _ptr(out["n_a"]), _ptr(out["matches_b"]), _ptr(out["n_b"]))
    return st, out


def test_capacity(FE):
    """More maxima than max_keypoints: fe_batch_run(sync), fe_batch_download and fe_pipeline_batch return FE_ERR_CAPACITY
    and n_kps reports the maxima found (upright, 4 octaves at 480x360: SURF drops nothing, so they are the survivors a
    large enough ctx holds)."""
    P = 2
    surf = dict(upright=True)
    Ls, Rs = synth.stereo_batch(H, W, P, seed0=29)
    with FE.FrontEnd(max_width=W, max_height=H, max_pairs=P, max_keypoints=8192) as f:
        f.set_batch_detector(surf)
        want = _batch(f, Ls, Rs, _cfg_a(FE), _cfg_b(FE))["n_kps"].copy()
    assert want.min() > 300
    with FE.FrontEnd(max_width=W, max_height=H, max_pairs=P, max_keypoints=256) as f:
        f.set_batch_detector(surf)
        f.batch_upload(Ls, Rs)
        with pytest.raises(FE.FeError) as e:
            f.batch_run(_cfg_a(FE), _cfg_b(FE), sync=True)
        assert e.value.code == FE.lib.FE_ERR_CAPACITY
        st, out = _raw_download(f, P)
        assert st == FE.lib.FE_ERR_CAPACITY and np.array_equal(out["n_kps"], want), (out["n_kps"], want)
        with pytest.raises(FE.FeError) as e:
            f.pipeline_batch(Ls, Rs, _cfg_a(FE), _cfg_b(FE))
        assert e.value.code == FE.lib.FE_ERR_CAPACITY


def test_full_size_batch(FE):
    """1280x720, 8 pairs, cv::SURF's defaults (threshold 100, 4 octaves, 2 layers, oriented SURF-64): every image equals
    fe_surf_detect_batch in raster order, both modes equal fe_stereo_match bit for bit, and the numpy matcher agrees on
    the first pair."""
    h, w, P = 720, 1280, 8
    Ls, Rs = synth.stereo_batch(h, w, P, seed0=0)
    with FE.FrontEnd(max_width=w, max_height=h, max_pairs=P) as f:
        f.set_batch_detector({})
        out = _batch(f, Ls, Rs, _cfg_a(FE), _cfg_b(FE))
        out = {k: v.copy() for k, v in out.items()}
        print("keypoints per image:", out["n_kps"].tolist(), "mode A:", out["n_a"].tolist(), "mode B:", out["n_b"].tolist())
        assert out["n_kps"].min() > 5000
        _check_against_single_entry(f, {}, Ls, Rs, out)
        _check_matches(FE, f, {}, out, P, 1)
