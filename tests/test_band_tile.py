"""The epipolar band kernel (hamming_band_tile_kernel, match.cu) against the oracle on inputs built to reach its edges.

A CTA takes 256 consecutive query indices, one per thread, stages the trains of [min lo, max hi) of their row-table ranges
in shared-memory chunks of 512 and has each thread test every train of its own range with the exact band predicate.  The
column arg-min of the inner band (mode B) meets in one shared-memory key per staged train and leaves with a global
atomicMin.  The cases here: spans of several chunks (one image row with more trains than a chunk holds), queries in any
order, empty and ragged sizes, fractional y with offsets and float32 |dy| exactly on the threshold, NORM_HAMMING2, and
column ties between queries on both sides of a 256-query block edge.  Every GPU test demands equal indices and distances.
"""
import numpy as np
import pytest

from oracle import match as omatch
from test_hamming_exhaustive import (CROSS_LAUNCHES, _assert_same, _flip, _kps, bits_hamming2, bits_random, bits_spread,
                                     bits_tight_lb4)

BLOCK, CHUNK = 256, 512                  # queries per CTA, trains per shared-memory chunk (match.cu BT_Q, BT_T)


@pytest.fixture(scope="module")
def FE(fe):
    return fe


def _step(x, k):
    """float32 x moved k representable steps."""
    x = np.float32(x)
    for _ in range(abs(k)):
        x = np.nextafter(x, np.float32(np.inf if k > 0 else -np.inf))
    return x


def edge_partner(ty, m, qoff, toff, sign, outside=False):
    """Query y (float32) whose float32 |(qy + qoff) - (ty + toff)| is exactly m on the side `sign` of the train -- or, with
    outside=True, one float32 step further out; None if no nearby float does it."""
    m = np.float32(m)
    b = np.float32(np.float32(ty) + np.float32(toff))
    a0 = np.float32(b + np.float32(sign) * m)
    for da in range(-6, 7):
        a = _step(a0, da)
        if np.abs(np.float32(a - b)) == m and (a >= b) == (sign > 0):
            break
    else:
        return None
    if outside:
        a = _step(a, 1 if sign > 0 else -1)
    q0 = np.float32(a - np.float32(qoff))
    for dq in range(-6, 7):
        q = _step(q0, dq)
        if np.float32(q + np.float32(qoff)) == a:
            return q
    return None


def band_scene(seed, nq, nt, thr, qoff=0.0, toff=0.0, dense=0, h2=False, shuffle=False):
    """(qd, qy, td, ty) with raster-ordered trains at ~8 per image row and fractional y.  `dense` trains share one row (the
    span of a block there needs several chunks) and each of them has a query near-copy in that row.  Of the other queries,
    three in five are near copies of a train whose y + toff lies in [0, 0.3) -- where float32 steps are fine enough for a
    difference of exactly float32(0.7) -- with |dy| exactly on the threshold or one float32 step outside it; the rest are
    near copies of a random train inside the band, or unrelated.  A tenth of the trains duplicate their neighbour, y
    included (ties for best and second).  shuffle: queries in random order."""
    rng = np.random.default_rng(seed)
    flip = (lambda r, k: _flip(r, bits_hamming2(k, rng))) if h2 else (lambda r, k: _flip(r, bits_random(k, rng)))
    span = max(nt // 8, 4)
    n_low = min(nt - dense, max((nt - dense) // 8, 1)) if nt > dense else 0
    low = np.float32(rng.uniform(0, 0.3, n_low)) - np.float32(toff)
    rest = nt - dense - n_low
    ty = np.sort(np.concatenate([low, rng.integers(0, 8 * span, rest) / 8 + rng.uniform(0, 0.1, rest),
                                 np.full(dense, span / 2 + 0.25)]).astype(np.float32))
    td = rng.integers(0, 256, (nt, 32), dtype=np.uint8)
    if nt > 1:
        dup = np.nonzero(rng.random(nt - 1) < 0.1)[0] + 1
        td[dup], ty[dup] = td[dup - 1], ty[dup - 1]
    d_rows = np.nonzero(ty == np.float32(span / 2 + 0.25))[0] if dense else np.zeros(0, np.int64)
    low_rows = np.nonzero(np.abs(ty + np.float32(toff) - np.float32(0.15)) <= np.float32(0.16))[0]
    qd = np.zeros((nq, 32), np.uint8)
    qy = np.zeros(nq, np.float32)
    for i in range(nq):
        if i < len(d_rows):                  # the dense row: one near copy of each of its trains
            j = d_rows[i]
            qd[i] = flip(td[j], int(rng.integers(0, 12)))
            qy[i] = np.float32(np.float32(ty[j]) + np.float32(toff) - np.float32(qoff))
            continue
        if nt == 0:
            qd[i], qy[i] = rng.integers(0, 256, 32, dtype=np.uint8), rng.uniform(0, 50)
            continue
        kind = i % 5
        edge = kind < 3 and len(low_rows) > 0
        j = int(rng.choice(low_rows)) if edge else int(rng.integers(0, nt))
        qd[i] = flip(td[j], int(rng.integers(0, 24))) if kind < 4 else rng.integers(0, 256, 32, dtype=np.uint8)
        y = edge_partner(ty[j], thr, qoff, toff, 1 if i % 2 else -1, outside=kind == 2) if edge else None
        if y is None:
            y = np.float32(ty[j] + np.float32(toff) - np.float32(qoff) + np.float32(rng.uniform(-thr, thr)))
        qy[i] = y
    order = rng.permutation(nq) if shuffle else np.argsort(qy, kind="stable")
    return qd[order], qy[order], td, ty


def _knn_ref(qd, qy, td, ty, thr, qoff, toff, h2):
    D = (omatch.hamming2_matrix if h2 else omatch.hamming_matrix)(qd, td)
    oi, od, _ = omatch.knn2(D, omatch.epipolar_mask(qy, ty, thr, qoff, toff))
    return oi, od


def _check_modes(FE, f, qd, qy, td, ty, thr, qoff=0.0, toff=0.0, h2=False, what=()):
    """knnMatch and mode A (ratio 0.8) through stereo_match against the oracle; the kNN-2 stage takes the banded path."""
    norm = FE.NORM_HAMMING2 if h2 else FE.NORM_HAMMING
    cfg = FE.match_cfg(mask=FE.MASK_EPIPOLAR, epi_threshold=thr, q_y_offset=qoff, t_y_offset=toff, norm=norm, ratio=0.8)
    f.profile_reset()
    idx, dist = f.knnMatch(_kps(FE, qy), qd, _kps(FE, ty), td, cfg)
    assert f.stage_times()["hamming_knn2"][1] == 2, what
    oi, od = _knn_ref(qd, qy, td, ty, thr, qoff, toff, h2)
    assert np.array_equal(idx, oi) and np.array_equal(dist, od), what
    got = f.stereo_match(_kps(FE, qy), qd, _kps(FE, ty), td, cfg)
    want = omatch.stereo_match_ratio(qy, ty, qd, td, thr, 0.8, "hamming2" if h2 else "hamming", qoff, toff)
    _assert_same(got, want, ("mode A",) + tuple(what))


def _check_cross(FE, f, qd, qy, td, ty, max_dy, what=()):
    """Mode B alone (its band pass is the tile kernel with the inner band) against the oracle, on the pruned path."""
    f.profile_reset()
    got = f.stereo_match(_kps(FE, qy), qd, _kps(FE, ty), td, FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE,
                                                                            max_dy=max_dy))
    assert f.stage_times()["hamming_cross"][1] == CROSS_LAUNCHES["join"], what
    _assert_same(got, omatch.stereo_match_crosscheck(qy, ty, qd, td, max_dy), ("mode B",) + tuple(what))


# ---- CPU: the generator does what it says ----------------------------------------------------------------------------
@pytest.mark.parametrize("qoff,toff", [(0.0, 0.0), (0.375, -1.25), (-0.1, 0.3)])
@pytest.mark.parametrize("thr", [0.0, 0.7, 2.0])
def test_band_scene_hits_the_threshold_exactly(thr, qoff, toff):
    qd, qy, td, ty = band_scene(3, 600, 700, thr, qoff, toff)
    assert np.all(np.diff(ty) >= 0) and np.all(np.diff(qy) >= 0)
    dy = np.abs((qy + np.float32(qoff))[:, None] - (ty + np.float32(toff))[None, :])
    m = np.float32(thr)
    assert (dy == m).sum() >= 100                                             # on the threshold: inside
    assert ((dy > m) & (dy < m + np.float32(1e-4))).sum() >= 50              # one float32 step above it: outside
    oi, od = _knn_ref(qd, qy, td, ty, thr, qoff, toff, False)
    best_on_edge = [i for i in range(len(qd)) if oi[i, 0] >= 0 and dy[i, oi[i, 0]] == m]
    assert len(best_on_edge) >= 50                                            # the boundary train is often the best one
    assert np.any((oi[:, 1] >= 0) & (od[:, 0] == od[:, 1]))                   # ties for best and second


def test_band_scene_dense_row_spans_several_chunks():
    qd, qy, td, ty = band_scene(4, 1600, 1700, 2.0, dense=1600)
    u, c = np.unique(ty, return_counts=True)
    row = ty == u[c.argmax()]
    assert row.sum() == 1600 and row.sum() // CHUNK == 3 and row.sum() % CHUNK > 0   # 3 full chunks and a partial one
    assert np.all(qy == u[c.argmax()])
    D = omatch.hamming_matrix(qd, td)
    assert np.all(D[:1600][np.arange(1600), np.nonzero(row)[0][:1600]] < 12)  # a near copy of every train of the row


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_multi_chunk_spans_vs_oracle(FE):
    """One image row with 1500 .. 4000 trains: every block of queries in that row stages its span in several 512-train
    chunks, the last one partial; counts up to 4097 and in any order; modes A and B."""
    cases = [(1600, 1700, 1600), (4097, 4097, 2100), (300, 4097, 4000), (4097, 1501, 1501)]
    with FE.FrontEnd(max_keypoints=4097, max_height=2048) as f:
        for i, (nq, nt, dense) in enumerate(cases):
            for thr in (2.0, 0.7):
                for shuffle in (False, True):
                    qd, qy, td, ty = band_scene(100 + i, nq, nt, thr, dense=dense, shuffle=shuffle)
                    _check_modes(FE, f, qd, qy, td, ty, thr, what=(nq, nt, thr, shuffle))
                    if not shuffle:
                        _check_cross(FE, f, qd, qy, td, ty, thr, what=(nq, nt, thr))


@pytest.mark.gpu
@pytest.mark.parametrize("thr", [0.0, 0.7, 2.0])
def test_shuffled_queries_vs_oracle(FE, thr):
    """Queries in random order against raster-ordered trains still take the banded path (2 launches); a block's span then
    covers most of the train list, which no first-and-last-query bound would."""
    with FE.FrontEnd(max_keypoints=4097, max_height=2048) as f:
        for i, (nq, nt) in enumerate([(1000, 1200), (4097, 4097), (257, 3000)]):
            qd, qy, td, ty = band_scene(200 + i, nq, nt, thr, shuffle=True)
            assert np.any(np.diff(qy) < 0)
            _check_modes(FE, f, qd, qy, td, ty, thr, what=(nq, nt, thr))


@pytest.mark.gpu
def test_empty_single_and_ragged_sizes(FE):
    sizes = [(0, 0), (0, 40), (40, 0), (1, 1), (1, 300), (300, 1), (255, 300), (256, 256), (257, 300), (513, 700),
             (1000, 999)]
    with FE.FrontEnd(max_keypoints=1024, max_height=2048) as f:
        for i, (nq, nt) in enumerate(sizes):
            for thr in (0.7, 2.0):
                qd, qy, td, ty = band_scene(300 + i, nq, nt, thr)
                _check_modes(FE, f, qd, qy, td, ty, thr, what=(nq, nt, thr))
                _check_cross(FE, f, qd, qy, td, ty, thr, what=(nq, nt, thr))


@pytest.mark.gpu
@pytest.mark.parametrize("qoff,toff", [(0.375, -1.25), (-0.1, 0.3), (0.0, 0.0)])
@pytest.mark.parametrize("thr", [0.0, 0.7, 2.0])
def test_offsets_and_threshold_edges(FE, thr, qoff, toff):
    """Fractional y, nonzero q_y_offset / t_y_offset, epi_threshold 0, and float32 |dy| exactly on the threshold (inside) and
    one step above it (outside)."""
    with FE.FrontEnd(max_keypoints=4096, max_height=2048) as f:
        for i, (nq, nt) in enumerate([(600, 700), (3000, 2500)]):
            qd, qy, td, ty = band_scene(400 + i, nq, nt, thr, qoff, toff)
            _check_modes(FE, f, qd, qy, td, ty, thr, qoff, toff, what=(nq, nt, thr, qoff, toff))


@pytest.mark.gpu
@pytest.mark.parametrize("thr", [0.0, 0.7, 2.0])
def test_hamming2_vs_oracle(FE, thr):
    with FE.FrontEnd(max_keypoints=4096, max_height=2048) as f:
        for i, (nq, nt, dense, shuffle) in enumerate([(700, 800, 0, False), (1600, 1700, 1600, False), (1000, 1200, 0, True)]):
            qd, qy, td, ty = band_scene(500 + i, nq, nt, thr, 0.25, -0.5, dense=dense, h2=True, shuffle=shuffle)
            _check_modes(FE, f, qd, qy, td, ty, thr, 0.25, -0.5, h2=True, what=(nq, nt, thr, shuffle))


def block_edge_ties(seed, n_blocks=6, max_dy=0.7):
    """Mode B scenario: at every 256-query block edge e, queries e - 1 and e are identical rows near train t, both in t's
    inner band, so the pair (e - 1, t) is mutual only if t's column key breaks the tie between two CTAs by index.  The
    other queries and trains are unrelated rows in rows of their own."""
    rng = np.random.default_rng(seed)
    nq = n_blocks * BLOCK
    qd = rng.integers(0, 256, (nq, 32), dtype=np.uint8)
    qy = np.repeat(np.arange(nq // 4, dtype=np.float32) * np.float32(3), 4)        # 4 queries per row, rows 3 apart
    td, ty = [], []
    for e in range(BLOCK, nq, BLOCK):
        qy[e - 2:e + 2] = qy[e]                                                     # e - 1 and e share a row
        qd[e] = qd[e - 1]
        row = qy[e]
        td.append(_flip(qd[e - 1], bits_tight_lb4(5, rng)))
        ty.append(np.float32(row + np.float32(0.5) * np.float32(max_dy)) if e % (2 * BLOCK) else row)
        td.append(_flip(rng.integers(0, 256, 32, dtype=np.uint8), bits_spread(3, rng)))
        ty.append(np.float32(row + np.float32(0.25)))
    for r in range(0, nq // 4, 7):                                                  # unrelated trains elsewhere
        td.append(rng.integers(0, 256, 32, dtype=np.uint8))
        ty.append(np.float32(3 * r + 1.5))
    o = np.argsort(np.array(ty, np.float32), kind="stable")
    return qd, qy, np.stack(td)[o], np.array(ty, np.float32)[o]


@pytest.mark.gpu
def test_column_tie_across_block_edge(FE):
    """Mode B without mode A: the column key of a train whose tied queries sit in two CTAs goes to the lower index."""
    for max_dy in (0.7, 2.0):
        qd, qy, td, ty = block_edge_ties(7, max_dy=max_dy)
        D = omatch.hamming_matrix(qd, td)
        q, t, _ = omatch.stereo_match_crosscheck(qy, ty, qd, td, max_dy)
        edges = np.arange(BLOCK, len(qd), BLOCK)
        assert np.all(np.isin(edges - 1, q)) and not np.any(np.isin(edges, q))     # the lower index wins every tie
        assert np.all(D[edges - 1] == D[edges])
        with FE.FrontEnd(max_keypoints=2048, max_height=2048) as f:
            for _ in range(3):
                _check_cross(FE, f, qd, qy, td, ty, max_dy, what=("edge ties", max_dy))
