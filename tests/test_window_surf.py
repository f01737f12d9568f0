"""SURF landmarks tracked across frames on the device: fe_window_batch, fe_window_update and fe_batch_landmarks on SURF-64 /
SURF-128 float rows matched with FE_NORM_L2.

The window kernels are the stereo matcher's own (banded or masked all-pairs FP32 kNN-2 + Lowe for WindowMatcher, the exact
all-pairs FP32 pass twice for liveGraph), so every batched track is demanded bit for bit equal to the host entry points
(fe_window_match, fe_stereo_match) on the same landmark rows, and within the north-star tolerance of the numpy oracle
(>= 99.9 % index agreement; the oracle's L2 is evaluated in float64, not in the device's FP32 order).
"""
import numpy as np
import pytest

from oracle import match as omatch
from oracle import synth

pytestmark = pytest.mark.gpu

H, W = 240, 320
KINDS = [("DESC_SURF128", 128), ("DESC_SURF64", 64)]


@pytest.fixture(scope="module")
def FE(fe):
    return fe


def _sequence(h, w, seed, n_frames):
    fr = synth.stereo_sequence(h, w, seed, n_frames)
    return np.stack([p[0] for p in fr]), np.stack([p[1] for p in fr])


def _surf_batch(FE, f, kind, Ls, Rs):
    """SURF features of the sequence with stereo ratio matching on the epipolar band (BASELINE config 3's cfg_a)."""
    f.set_batch_descriptor(getattr(FE, kind))
    return f.pipeline_batch(Ls, Rs, FE.match_cfg(norm=FE.NORM_L2), None)


def _landmarks(out, fr):
    """(left kps, left rows, right kps, right rows) of frame fr: every stereo ratio match is a landmark."""
    m = out["matches_a"][fr][:out["n_a"][fr]]
    return (out["kps"][2 * fr][m["queryIdx"]], out["desc"][2 * fr][m["queryIdx"]],
            out["kps"][2 * fr + 1][m["trainIdx"]], out["desc"][2 * fr + 1][m["trainIdx"]])


def _xy(k):
    return np.stack([k["x"], k["y"]], 1)


def _same_bits(a, b):
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def _window_cfg(FE):
    return FE.match_cfg(mask=FE.MASK_WINDOW, norm=FE.NORM_L2)


def _live_cfg(FE):
    return FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, norm=FE.NORM_L2)


def _host_live(FE, f, kind, cur, prev):
    """liveGraph on the host entry point: fe_stereo_match cross-check (no mask, no |dy| filter) of the left rows and of the
    right rows, intersected on the same previous landmark."""
    cc = FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, norm=FE.NORM_L2, max_dy=-1.0)
    ml = f.stereo_match(cur[0], cur[1], prev[0], prev[1], cc, kind=getattr(FE, kind))
    mr = f.stereo_match(cur[2], cur[3], prev[2], prev[3], cc, kind=getattr(FE, kind))
    right = dict(zip(mr["queryIdx"].tolist(), mr["trainIdx"].tolist()))
    keep = np.array([right.get(q, -1) == t for q, t in zip(ml["queryIdx"].tolist(), ml["trainIdx"].tolist())], bool)
    return ml[keep]


class Agreement:
    """Oracle tracks the device reproduces (same query, same train; distance within rtol 1e-5), summed over frame pairs."""

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


@pytest.mark.parametrize("kind,dim", KINDS)
def test_window_batch_surf_matches_host_and_oracle(FE, kind, dim):
    """WindowMatcher over a resident 10-frame SURF sequence (box mask on the left coordinates, left rows, kNN-2, Lowe 0.8):
    bit for bit the host fe_window_match on the landmark rows downloaded from the batch, >= 99.9 % of the oracle's tracks;
    triangulation against numpy in double; fe_batch_landmarks returns the float rows bit for bit."""
    F, N = 10, 400
    Ls, Rs = _sequence(H, W, 41, F)
    Q = np.array([[1, 0, 0, -160.5], [0, 1, 0, -120.25], [0, 0, 0, 420.0], [0, 0, 1.0 / 0.12, 0]], np.float64)
    with FE.FrontEnd(max_width=W, max_height=H, max_pairs=F, max_keypoints=1024, n_features=N, orientation=False,
                     surf_upright=True) as f:
        out = _surf_batch(FE, f, kind, Ls, Rs)
        tracks, n_tr, xyz = f.window_batch(Q=Q)
        # stereoLandmarks packing of the same resident batch, before any host call reuses the context's device slots
        pk = f.batch_landmarks(0)
        lm = [_landmarks(out, fr) for fr in range(F)]
        assert pk["l_desc"].dtype == np.float32 and pk["l_desc"].shape[2] == dim and pk["r_desc"].shape[2] == dim
        for fr in range(F):
            m = out["matches_a"][fr][:out["n_a"][fr]]
            n = len(m)
            assert pk["n"][fr] == n
            assert np.array_equal(pk["l_kps"][fr][:n], lm[fr][0]) and np.array_equal(pk["r_kps"][fr][:n], lm[fr][2])
            assert _same_bits(pk["l_desc"][fr][:n], lm[fr][1]) and _same_bits(pk["r_desc"][fr][:n], lm[fr][3])
            pm = pk["matches"][fr][:n]
            assert np.array_equal(pm["queryIdx"], np.arange(n)) and np.array_equal(pm["trainIdx"], np.arange(n))
            assert _same_bits(pm["distance"], m["distance"]) and np.all(pm["imgIdx"] == 0)
        agree = Agreement()
        for fr in range(1, F):
            got = tracks[fr - 1][:n_tr[fr - 1]]
            cur, prev = lm[fr], lm[fr - 1]
            assert len(got) > 100
            one = f.window_match(cur[0], cur[1], prev[0], prev[1], cfg=_window_cfg(FE), kind=getattr(FE, kind))
            assert _same_bits(one, got), fr
            agree.add(got, *omatch.window_match(_xy(cur[0]), _xy(prev[0]), cur[1], prev[1], norm="l2"))
        agree.check()
    for fr in (0, 5, 9):
        lk, rk = lm[fr][0], lm[fr][2]
        inp = np.stack([lk["x"].astype(np.float64), lk["y"].astype(np.float64),
                        (lk["x"] - rk["x"]).astype(np.float64), np.ones(len(lk))], 0)
        hom = Q @ inp
        assert np.allclose(xyz[fr][:len(lk)], (hom[:3] / (1000.0 * hom[3])).T, rtol=1e-12, atol=0)


@pytest.mark.parametrize("kind,dim", KINDS)
def test_window_batch_surf_live_graph(FE, kind, dim):
    """liveGraph's tracker (algorithm.py:1160-1190) over a resident SURF sequence: no |dy| filter, cross-check of the left
    rows and of the right rows, same previous landmark.  Bit for bit two host fe_stereo_match cross-checks intersected on
    the host; >= 99.9 % of oracle.match.live_graph_tracks."""
    F, N = 6, 400
    Ls, Rs = _sequence(H, W, 47, F)
    with FE.FrontEnd(max_width=W, max_height=H, max_pairs=F, max_keypoints=1024, n_features=N, orientation=False,
                     surf_upright=True) as f:
        out = _surf_batch(FE, f, kind, Ls, Rs)
        tracks, n_tr, _ = f.window_batch(cfg=_live_cfg(FE))
        lm = [_landmarks(out, fr) for fr in range(F)]
        agree = Agreement()
        for fr in range(1, F):
            got = tracks[fr - 1][:n_tr[fr - 1]]
            assert len(got) > 100
            assert _same_bits(got, _host_live(FE, f, kind, lm[fr], lm[fr - 1])), fr
            agree.add(got, *omatch.live_graph_tracks(lm[fr][1], lm[fr - 1][1], lm[fr][3], lm[fr - 1][3], norm="l2"))
        agree.check()


@pytest.mark.parametrize("kind,dim", KINDS)
def test_window_update_surf_equals_batched_tracks(FE, kind, dim):
    """fe_window_update with SURF rows: per update bit for bit the batched tracks of the same frames, in WindowMatcher mode
    under the C++ window rule (nWindow = 3) and in liveGraph mode under the Python rule (length = 4), across a reset.
    Updates that mix row kinds without a reset, SURF with Hamming and ORB with L2 fail and leave the window unchanged."""
    F, N = 6, 400
    Ls, Rs = _sequence(H, W, 53, F)
    K = getattr(FE, kind)
    with FE.FrontEnd(max_width=W, max_height=H, max_pairs=F, max_keypoints=1024, n_features=N, orientation=False,
                     surf_upright=True) as f:
        out = _surf_batch(FE, f, kind, Ls, Rs)
        tr_a, n_a, _ = f.window_batch()
        tr_a = [t[:n].copy() for t, n in zip(tr_a, n_a)]
        tr_b, n_b, _ = f.window_batch(cfg=_live_cfg(FE))
        tr_b = [t[:n].copy() for t, n in zip(tr_b, n_b)]
        lm = [_landmarks(out, fr) for fr in range(F)]
        for fr in range(F):
            tr, frames = f.window_update(lm[fr][0], lm[fr][1], kind=K)
            assert frames == min(fr + 1, 2)
            assert len(tr) == 0 if fr == 0 else _same_bits(tr, tr_a[fr - 1]), fr
        tr, frames = f.window_update(reset=True)
        assert len(tr) == 0 and frames == 0
        for fr in range(F - 1):
            tr, frames = f.window_update(lm[fr][0], lm[fr][1], lm[fr][3], cfg=_live_cfg(FE), length=4, variant=1, kind=K)
            assert frames == min(fr + 1, 4)
            assert len(tr) == 0 if fr == 0 else _same_bits(tr, tr_b[fr - 1]), fr
        # failed updates: nothing of the window changes
        cur = lm[F - 1]
        other, odim = ("DESC_SURF64", 64) if dim == 128 else ("DESC_SURF128", 128)
        rows = np.ascontiguousarray(np.resize(cur[1], (len(cur[0]), odim)))
        for call, code in (
                (lambda: f.window_update(cur[0], rows, rows, cfg=_live_cfg(FE), length=4, variant=1, kind=getattr(FE, other)),
                 FE.lib.FE_ERR_BAD_ARG),
                (lambda: f.window_update(cur[0], np.zeros((len(cur[0]), 32), np.uint8), np.zeros((len(cur[0]), 32), np.uint8),
                                         cfg=FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE), length=4, variant=1),
                 FE.lib.FE_ERR_BAD_ARG),
                (lambda: f.window_update(cur[0], cur[1], cur[3], cfg=FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE),
                                         length=4, variant=1, kind=K), FE.lib.FE_ERR_UNSUPPORTED),
                (lambda: f.window_update(cur[0], np.zeros((len(cur[0]), 32), np.uint8), np.zeros((len(cur[0]), 32), np.uint8),
                                         cfg=_live_cfg(FE), length=4, variant=1), FE.lib.FE_ERR_UNSUPPORTED)):
            with pytest.raises(FE.FeError) as e:
                call()
            assert e.value.code == code
        with pytest.raises(ValueError):
            f.window_update(cur[0], cur[1].astype(np.float64), kind=K)
        tr, frames = f.window_update(cur[0], cur[1], cur[3], cfg=_live_cfg(FE), length=4, variant=1, kind=K)
        assert frames == 4 and _same_bits(tr, tr_b[F - 2])
        # binary rows after float rows, and float rows after binary rows, need a reset in between
        f.window_update(reset=True)
        f.window_update(cur[0], np.zeros((len(cur[0]), 32), np.uint8))
        with pytest.raises(FE.FeError) as e:
            f.window_update(cur[0], cur[1], kind=K)
        assert e.value.code == FE.lib.FE_ERR_BAD_ARG
        f.window_update(reset=True)
        tr, frames = f.window_update(cur[0], cur[1], kind=K)
        assert len(tr) == 0 and frames == 1
    # the sequence-level errors of fe_window_batch: Hamming on a SURF batch, L2 on an ORB batch
    with FE.FrontEnd(max_width=W, max_height=H, max_pairs=2, max_keypoints=1024, n_features=N) as f:
        _surf_batch(FE, f, kind, Ls[:2], Rs[:2])
        with pytest.raises(FE.FeError) as e:
            f.window_batch(cfg=FE.match_cfg(mask=FE.MASK_WINDOW))
        assert e.value.code == FE.lib.FE_ERR_UNSUPPORTED
        f.set_batch_descriptor(FE.DESC_ORB256)
        f.pipeline_batch(Ls[:2], Rs[:2], FE.match_cfg(), None)
        with pytest.raises(FE.FeError) as e:
            f.window_batch(cfg=_window_cfg(FE))
        assert e.value.code == FE.lib.FE_ERR_UNSUPPORTED


def _l2_exact(a, b):
    """L2 distances by explicit differences in float64 (no |a|^2 + |b|^2 - 2ab expansion): identical rows give identical
    distances, so exact duplicates tie exactly as they do on the device."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    out = np.empty((len(a), len(b)), np.float32)
    for s in range(0, len(a), 32):
        out[s:s + 32] = np.sqrt(((a[s:s + 32, None, :] - b[None, :, :]) ** 2).sum(-1))
    return out


@pytest.mark.parametrize("kind,dim", KINDS)
def test_window_update_surf_duplicate_rows_resolve_to_lower_train(FE, kind, dim):
    """Exact duplicates of previous landmarks (keypoint and both rows), planted right after the original inside the box:
    kNN-2 reports the lower train index first and Lowe rejects the tie; the cross-check keeps the lower train index -- as the
    oracle's first-minimum rules do on the same rows."""
    F, N = 2, 400
    Ls, Rs = _sequence(H, W, 59, F)
    K = getattr(FE, kind)
    with FE.FrontEnd(max_width=W, max_height=H, max_pairs=F, max_keypoints=1024, n_features=N, orientation=False,
                     surf_upright=True) as f:
        out = _surf_batch(FE, f, kind, Ls, Rs)
        cur, prev = _landmarks(out, 1), _landmarks(out, 0)
        planted = np.arange(0, len(prev[0]), 7)
        at = planted + 1
        prev = tuple(np.insert(a, at, a[planted], axis=0) for a in prev)
        orig = planted + np.arange(len(planted))          # positions of the originals after the insertion
        dups = orig + 1
        assert np.all(np.diff(prev[0]["y"]) >= 0)           # still raster-ordered: the banded kernel runs
        Dl, Dr = _l2_exact(cur[1], prev[1]), _l2_exact(cur[3], prev[3])
        # kNN-2 on the host entry point: the original comes first, its duplicate second, at the same distance
        idx, dist = f.knnMatch(cur[0], cur[1], prev[0], prev[1], _window_cfg(FE), kind=K)
        tie = np.isin(idx[:, 0], orig)
        assert tie.sum() > 10 and np.array_equal(idx[tie, 1], idx[tie, 0] + 1) and _same_bits(dist[tie, 0], dist[tie, 1])
        assert not np.isin(idx[:, 0], dups).any()
        oi, od, _ = omatch.knn2(Dl, omatch.window_mask(cur[0]["x"], cur[0]["y"], prev[0]["x"], prev[0]["y"]))
        otie = np.isin(oi[:, 0], orig)
        assert np.array_equal(oi[otie, 1], oi[otie, 0] + 1) and not np.isin(oi[:, 0], dups).any()
        assert (otie != tie).sum() <= 1 and np.array_equal(oi[tie & otie], idx[tie & otie])
        # WindowMatcher: the ties are rejected by the ratio test, on the device and in the oracle
        f.window_update(prev[0], prev[1], kind=K)
        tr, _ = f.window_update(cur[0], cur[1], kind=K)
        assert len(tr) > 100 and _same_bits(tr, f.window_match(cur[0], cur[1], prev[0], prev[1], cfg=_window_cfg(FE), kind=K))
        q, _, _ = omatch.lowe_ratio(oi, od, 0.8)
        assert not np.isin(tr["queryIdx"], np.nonzero(tie)[0]).any() and not np.isin(q, np.nonzero(otie)[0]).any()
        # liveGraph: mutual on both sides with the lower train index
        f.window_update(reset=True)
        f.window_update(prev[0], prev[1], prev[3], cfg=_live_cfg(FE), kind=K)
        tr, _ = f.window_update(cur[0], cur[1], cur[3], cfg=_live_cfg(FE), kind=K)
        assert _same_bits(tr, _host_live(FE, f, kind, cur, prev))
        ql, tl, _ = omatch.cross_check(Dl)
        qr, tr_, _ = omatch.cross_check(Dr)
        right = dict(zip(qr.tolist(), tr_.tolist()))
        keep = np.array([right.get(a, -1) == b for a, b in zip(ql.tolist(), tl.tolist())], bool)
        ql, tl = ql[keep], tl[keep]
        assert not np.isin(tr["trainIdx"], dups).any() and not np.isin(tl, dups).any()
        on_planted = np.isin(tr["trainIdx"], orig)
        assert on_planted.sum() > 10
        want = dict(zip(ql.tolist(), tl.tolist()))
        assert sum(want.get(a) != b for a, b in zip(tr["queryIdx"][on_planted].tolist(), tr["trainIdx"][on_planted].tolist())) <= 1


@pytest.mark.parametrize("kind,dim", KINDS)
def test_window_batch_surf_pyramid_landmarks(FE, kind, dim):
    """With fe_set_orb_pyramid(3, 1.2) the landmarks are level-major, not raster-ordered: the window runs the masked
    all-pairs FP32 kernel (one launch, where the banded path takes a row table and a band launch) and its tracks equal the
    host matcher's bit for bit."""
    F, N = 4, 500
    Ls, Rs = _sequence(H, W, 43, F)
    with FE.FrontEnd(max_width=W, max_height=H, max_pairs=F, max_keypoints=2048, n_features=N, surf_upright=True) as f:
        f.set_pyramid(3, 1.2)
        out = _surf_batch(FE, f, kind, Ls, Rs)
        before = f.stage_times()["l2_match_fp32"][1]
        tracks, n_tr, _ = f.window_batch()
        assert f.stage_times()["l2_match_fp32"][1] - before == 1
        lm = [_landmarks(out, fr) for fr in range(F)]
        for fr in range(1, F):
            cur, prev = lm[fr], lm[fr - 1]
            assert (np.diff(prev[0]["y"]) < 0).any() and (prev[0]["octave"] > 0).any()
            got = tracks[fr - 1][:n_tr[fr - 1]]
            assert len(got) > 50
            one = f.window_match(cur[0], cur[1], prev[0], prev[1], cfg=_window_cfg(FE), kind=getattr(FE, kind))
            assert _same_bits(one, got), fr


def test_window_batch_surf128_full_size(FE):
    """Config 4's shape with SURF-128 features (10 frames of 1280x720, N = 5000 FAST keypoints, upright SURF_EXTENDED, ratio
    band stereo matching): tracks ordered by queryIdx, inside the 100x100 search box, and the synthetic camera step
    recovered as a (-3, -1) px landmark motion by most tracks (measured on a B200 at 1000 W: 0.962 to 0.968 of every frame
    pair's ~4050 tracks; the bound leaves a margin below that)."""
    h, w, F, N = 720, 1280, 10, 5000
    Ls, Rs = _sequence(h, w, 7, F)
    with FE.FrontEnd(max_width=w, max_height=h, max_pairs=F, max_keypoints=8192, n_features=N, orientation=False,
                     surf_upright=True) as f:
        out = _surf_batch(FE, f, "DESC_SURF128", Ls, Rs)
        tracks, n_tr, _ = f.window_batch()
    shares = []
    for fr in range(1, F):
        t = tracks[fr - 1][:n_tr[fr - 1]]
        (ck, _, _, _), (pk, _, _, _) = _landmarks(out, fr), _landmarks(out, fr - 1)
        assert len(t) > 1000 and np.all(np.diff(t["queryIdx"].astype(np.int64)) > 0)
        dx, dy = ck["x"][t["queryIdx"]] - pk["x"][t["trainIdx"]], ck["y"][t["queryIdx"]] - pk["y"][t["trainIdx"]]
        assert np.all(np.abs(dx) < 50) and np.all(np.abs(dy) < 50)
        shares.append(float(np.mean((dx == -3) & (dy == -1))))
    print("share of (-3, -1) px tracks per frame pair:", ["%.4f" % s for s in shares], "tracks:", list(n_tr))
    assert min(shares) > 0.9
