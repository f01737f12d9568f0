"""Hamming matchers against brute force on descriptors built to sit on the edges of the pruned cross-check.

Mode B on raster-ordered keypoints (launch_hamming_cross_pruned, match.cu) does not compare every pair: it takes band
candidates, sorts the entries into classes A / B / C / D by their candidate distance d* (splits 15, 24, 48), settles A x A
with a multi-index hash join over 16-bit halves, skips pairs by the lower bounds LB4 / LB8 (popcount of the OR of the xor
words) and runs several verification launches, some with queries and trains swapped.  Each step is exact on paper; a
`<` for a `<=` or a class split off by one loses a few pairs only, and natural-image descriptors seldom sit on those edges.

The generators below plant pairs at exact distances and control where the differing bits are, so that the join's
pigeonhole is tight, LB4 or LB8 equals the distance, ties cross the |dy| band edge at lower and higher indices, and
float32 |qy - ty| lands exactly on max_dy.  The CPU tests check that the generators do what they say; the GPU tests
demand bit-exact queryIdx / trainIdx / distance against the oracle for every path (and check which path ran), the
tuning knobs, the batched pipeline on images with tiled texture, and the kNN-2 / ratio edges.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import match as omatch

ROOT_DIR = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

D_STAR = (0, 1, 14, 15, 16, 17, 23, 24, 25, 47, 48, 49, 64, 128)    # both sides of every class split
MAX_DY = (0.0, 0.7, 2.0, 4096.0)                                      # 4096 exceeds every y range used here
# hamming_cross stage launches of each path ("fused": the batched pipeline's, whose band pass ran in mode A's stage)
CROSS_LAUNCHES = {"all_pairs": 1, "scan": 8, "join": 11, "fused_scan": 7, "fused_join": 10}


@pytest.fixture(scope="module")
def FE(fe):
    return fe


# ---- 1. descriptor generators with known structure ---------------------------------------------------------------------
def _flip(row, bits):
    w = np.ascontiguousarray(row).view("<u4").copy()
    for b in np.asarray(bits, np.int64):
        w[b // 32] ^= np.uint32(1 << int(b % 32))
    return w.view(np.uint8)


def bits_spread(k, rng):
    """k <= 16 bits, at most one per 16-bit half (k = 15: exactly one half identical; k = 16: none)."""
    halves = rng.choice(16, k, replace=False)
    return 16 * halves + rng.integers(0, 16, k)


def bits_tight_lb4(k, rng):
    """k <= 32 bits in words 0 .. 3 at distinct positions mod 32: LB4 = LB8 = d."""
    return 32 * rng.integers(0, 4, k) + rng.choice(32, k, replace=False)


def bits_tight_lb8(k, rng):
    """k <= 64 bits, distinct positions mod 32 within words 0 .. 3 and within words 4 .. 7: LB8 = d."""
    k1 = min(32, max(k - 32, (k + 1) // 2))
    lo = 32 * rng.integers(0, 4, k1) + rng.choice(32, k1, replace=False)
    hi = 128 + 32 * rng.integers(0, 4, k - k1) + rng.choice(32, k - k1, replace=False)
    return np.concatenate([lo, hi])


def bits_concentrated(k, rng):
    """k <= 32 bits, all in one word."""
    return 32 * int(rng.integers(0, 8)) + rng.choice(32, k, replace=False)


def bits_random(k, rng):
    return rng.choice(256, k, replace=False)


BITS = {"spread": (bits_spread, 16), "tight4": (bits_tight_lb4, 32), "tight8": (bits_tight_lb8, 64),
        "concentrated": (bits_concentrated, 32), "random": (bits_random, 256)}


def planted(kind, n, k, rng):
    """(q_desc, t_desc): n random rows and the same rows with k bits flipped by the `kind` pattern."""
    q = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    t = np.stack([_flip(r, BITS[kind][0](k, rng)) for r in q]) if n else q.copy()
    return q, t


def bits_hamming2(k, rng):
    """Bits of k distinct two-bit symbols; a symbol changes one or both of its bits (both kinds once k >= 3)."""
    sym = rng.choice(128, k, replace=False)
    how = rng.integers(1, 4, k)
    if k >= 3:
        how[:3] = (1, 2, 3)
    return np.array([2 * s + b for s, h in zip(sym, how) for b in (0, 1) if h >> b & 1], np.int64)


def hamming2_planted(n, k, rng):
    """NORM_HAMMING2 pairs at exactly k differing two-bit symbols."""
    q = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    t = np.stack([_flip(r, bits_hamming2(k, rng)) for r in q]) if n else q.copy()
    return q, t


def duplicates(rng, copies=40):
    """Rows that repeat: one row many times, all-zero and all-ones rows, and rows that share 15 of their 16 halves with
    many others (long probe runs in the join's hash table)."""
    row = rng.integers(0, 256, 32, dtype=np.uint8)
    near = np.repeat(rng.integers(0, 256, (1, 32), dtype=np.uint8), copies, axis=0)
    h = int(rng.integers(0, 16))
    near.view("<u2")[:, h] = rng.integers(0, 65536, copies, dtype=np.uint16)
    q = np.concatenate([np.repeat(row[None], copies, 0), np.zeros((copies // 4, 32), np.uint8),
                        np.full((copies // 4, 32), 255, np.uint8), near])
    t = q[rng.permutation(len(q))]
    return q, t


def unrelated(n, m, rng):
    return rng.integers(0, 256, (n, 32), dtype=np.uint8), rng.integers(0, 256, (m, 32), dtype=np.uint8)


def _lb(q, t, words):
    x = np.bitwise_xor(np.ascontiguousarray(q).view("<u4")[:, words], np.ascontiguousarray(t).view("<u4")[:, words])
    return np.bitwise_count(np.bitwise_or.reduce(x, axis=1)).astype(np.int64)


def _lb4(q, t):
    return _lb(q, t, slice(0, 4))


def _lb8(q, t):
    return _lb(q, t, slice(0, 4)) + _lb(q, t, slice(4, 8))


def _diag(q, t):
    return np.array([omatch.hamming_matrix(a[None], b[None])[0, 0] for a, b in zip(q, t)], np.int64)


@pytest.mark.parametrize("k", [0, 1, 7, 15, 16])
def test_spread_generator(k):
    q, t = planted("spread", 64, k, np.random.default_rng(k))
    assert np.all(_diag(q, t) == k)
    same = q.view("<u2") == t.view("<u2")
    assert np.all(same.sum(1) == 16 - k)                                     # k = 15: one identical half, 16: none
    assert np.all(np.bitwise_count(q.view("<u2") ^ t.view("<u2")) <= 1)     # at most one differing bit per half


@pytest.mark.parametrize("kind,ks", [("tight4", (0, 1, 14, 15, 16, 24, 25, 32)), ("tight8", (0, 25, 47, 48, 49, 64)),
                                     ("concentrated", (1, 15, 24, 32)), ("random", (64, 128))])
def test_planted_generators_have_exact_distance_and_tight_bounds(kind, ks):
    rng = np.random.default_rng(len(kind))
    for k in ks:
        q, t = planted(kind, 48, k, rng)
        assert np.all(_diag(q, t) == k), (kind, k)
        if kind == "tight4":
            assert np.all(_lb4(q, t) == k) and np.array_equal(q[:, 16:], t[:, 16:])
        if kind == "tight8":
            assert np.all(_lb8(q, t) == k)
        if kind == "concentrated":
            assert np.all((q.view("<u4") != t.view("<u4")).sum(1) == (1 if k else 0))
        assert np.all(_lb4(q, t) <= _diag(q, t)) and np.all(_lb8(q, t) <= _diag(q, t))


def test_hamming2_generator_counts_symbols():
    rng = np.random.default_rng(2)
    for k in (0, 1, 3, 8, 40):
        q, t = hamming2_planted(32, k, rng)
        d2 = np.array([omatch.hamming2_matrix(a[None], b[None])[0, 0] for a, b in zip(q, t)])
        d1 = _diag(q, t)
        assert np.all(d2 == k) and np.all((d1 >= k) & (d1 <= 2 * k))
        if k >= 3:
            assert np.all(d1 > k)                    # some symbols changed both bits and still count once


def test_duplicates_and_unrelated_generators():
    rng = np.random.default_rng(4)
    q, t = duplicates(rng)
    D = omatch.hamming_matrix(q, t)
    assert (D == 0).sum(1).max() >= 40                                       # one row repeated 40 times
    assert np.any(np.all(q == 0, 1)) and np.any(np.all(q == 255, 1))
    halves = q.view("<u2")
    share15 = ((halves[:, None, :] == halves[None, :, :]).sum(2) >= 15).sum(1)
    assert share15.max() >= 40
    a, b = unrelated(300, 300, rng)
    assert omatch.hamming_matrix(a, b).min() > 64                           # every candidate would be class D


# ---- 2. scenario builder for the cross-check ---------------------------------------------------------------------------
def _y_pair(base, target, side):
    """(qy, ty) float32 near `base` with float32 |qy - ty| == target (side 0), the nearest representable difference above
    it (side 1) or below it (side -1)."""
    ty = np.float32(base)
    qy0 = np.float32(ty + np.float32(target))
    best = None
    for k in range(-8, 9):
        qy = qy0
        for _ in range(abs(k)):
            qy = np.nextafter(qy, np.float32(np.inf if k > 0 else -np.inf))
        diff = np.abs(qy - ty)
        ok = diff == target if side == 0 else (diff > target if side > 0 else diff < target)
        if ok and (best is None or abs(float(diff) - float(target)) < abs(float(best[0]) - float(target))):
            best = (diff, qy)
    return None if best is None else (best[1], ty)


class _Builder:
    def __init__(self):
        self.q, self.t = [], []                       # (y, order, desc)

    def add(self, side, y, desc):
        lst = self.q if side == 0 else self.t
        lst.append((np.float32(y), len(lst), np.asarray(desc, np.uint8)))

    def finish(self, nq, nt):
        out = []
        for lst, n in ((self.q, nq), (self.t, nt)):
            lst = sorted(lst, key=lambda e: (e[0], e[1]))[:n]          # raster order; equal y keeps insertion order
            y = np.array([e[0] for e in lst], np.float32)
            d = np.stack([e[2] for e in lst]) if lst else np.zeros((0, 32), np.uint8)
            out += [d, y]
        return out


def cross_scenario(nq, nt, max_dy, seed):
    """(qd, qy, td, ty): raster-ordered query and train sets built from planted groups, then background.

    A group plants (q0, t0) at d in D_STAR and adds some of: a train tied with t0 at a lower index outside q0's band, a
    train tied with t0 at a higher index inside it, the same two for the column (queries tied for t0), competitors at
    d - 1 outside and d + 1 inside the band, and own partners at a lower distance for the out-of-band competitors (so
    that their thresholds are below the tie).  The planted |dy| is 0, exactly max_dy in float32, one representable
    step above or below it, or fractional.  Background: entries with no band candidate, unrelated rows, duplicates."""
    rng = np.random.default_rng(seed)
    m = np.float32(max_dy)
    huge = max_dy > 100
    off = np.float32(1.5 if huge else 2 * m + 1.5)
    B = _Builder()
    groups = [(d, v) for d in D_STAR for v in range(6)]
    rng.shuffle(groups)
    Y = np.float32(0.0)
    if 0 < max_dy <= 100:
        # float32 |qy - ty| == max_dy exactly for a value like 0.7 needs the fine float steps of rows near y = 0
        for d in (15, 24, 48):
            q0 = rng.integers(0, 256, 32, dtype=np.uint8)
            B.add(0, m, q0)
            B.add(1, 0.0, _flip(q0, BITS["tight8"][0](d, rng)))
        Y = np.float32(m + off + 1)
    # class C: a planted pair (q0, t0) at 40 loses its column to an earlier query c at the same distance with LB8 == 40,
    # while c's own threshold is 30 -- only the LB8 test against t0's threshold can find c, and 40 class-C fillers keep
    # c's partner out of t0's warp.  (q1, t1) loses its row the same way to an earlier train c2.
    q0, q1 = rng.integers(0, 256, (2, 32), dtype=np.uint8)
    t0, t1 = _flip(q0, bits_random(40, rng)), _flip(q1, bits_random(40, rng))
    c, c2 = _flip(t0, bits_tight_lb8(40, rng)), _flip(q1, bits_tight_lb8(40, rng))
    B.add(0, Y, c)
    B.add(1, Y, _flip(c, bits_random(30, rng)))
    Y = np.float32(Y + off)
    B.add(1, Y, c2)
    B.add(0, Y, _flip(c2, bits_random(30, rng)))
    for i in range(40):
        Y = np.float32(Y + off)
        f = rng.integers(0, 256, 32, dtype=np.uint8)
        B.add(0, Y, f)
        B.add(1, Y, _flip(f, bits_random(25 + i % 24, rng)))
    for qq, tt in ((q0, t0), (q1, t1)):
        Y = np.float32(Y + off)
        B.add(0, Y, qq)
        B.add(1, Y, tt)
    Y = np.float32(Y + off)
    kinds = [k for k in BITS]
    for d, v in groups:
        if len(B.q) >= nq and len(B.t) >= nt:
            break
        pat = [k for k in kinds if d <= BITS[k][1]]
        pat = pat[v % len(pat)]
        pb = lambda k: BITS[pat if k <= BITS[pat][1] else "random"][0](k, rng)
        q0 = rng.integers(0, 256, 32, dtype=np.uint8)
        t0 = _flip(q0, pb(d))
        r_out, r0 = Y, np.float32(Y + off)
        dyk = ("zero", "eq", "below", "above", "frac", "eq")[v]
        yp = None
        if not huge and dyk in ("eq", "below", "above"):
            yp = _y_pair(r0, m, {"eq": 0, "above": 1, "below": -1}[dyk])
        if yp is None:
            yp = (r0, r0) if dyk != "frac" else (r0, np.float32(r0 + np.float32(min(float(m), 1.0)) * np.float32(0.5)))
        qy0, ty0 = yp
        if rng.random() < 0.5:
            qy0, ty0 = ty0, qy0
        B.add(0, qy0, q0)
        B.add(1, ty0, t0)
        mode = v % 3
        partner = v % 2 == 0
        if mode in (0, 2):                     # row: tie at a lower index outside the band
            c = _flip(q0, pb(d))
            B.add(1, r_out, c)
            if partner and d > 0:
                B.add(0, r_out, _flip(c, pb(d // 2)))
        if mode in (1, 2):                     # column: tie at a lower index outside t0's band
            c = _flip(t0, pb(d))
            B.add(0, r_out, c)
            if partner and d > 0:
                B.add(1, r_out, _flip(c, pb(d // 2)))
        if mode == 0:                          # column tie inside the band at a higher index
            B.add(0, qy0, _flip(t0, pb(d)))
        if mode == 1:                          # row tie inside the band at a higher index
            B.add(1, ty0, _flip(q0, pb(d)))
        if d >= 1 and v in (1, 4):             # near competitors: d - 1 outside, d + 1 inside the band
            B.add(1, r_out, _flip(q0, pb(d - 1)))
            B.add(0, qy0, _flip(t0, pb(d + 1)))
        if v in (2, 5):
            B.add(0, r_out, _flip(t0, pb(d - 1)) if d >= 1 else t0)
            B.add(1, ty0, _flip(q0, pb(d + 1)))
        Y = np.float32(max(qy0, ty0) + off + 1.0)
    # background: lone entries (no band candidate), unrelated rows, duplicates, several keypoints per fractional row
    need = max(nq - len(B.q), nt - len(B.t), 0)
    if need:
        dq, dt = duplicates(rng, copies=max(8, min(64, need // 8)))
        rows = Y + off + np.sort(rng.integers(0, max(need // 4, 2), need + len(dq))).astype(np.float32) * np.float32(0.25)
        a, b = unrelated(need, need, rng)
        for i in range(0, need, 5):                # near copies in the same row: mutual matches at every index range
            b[i] = _flip(a[i], bits_random(i % 40, rng))
        for i in range(need):
            if len(B.q) < nq and not (i % 7 == 3):
                B.add(0, rows[i], a[i])
            if len(B.t) < nt and not (i % 7 == 5):
                B.add(1, rows[i] + np.float32(0.5) * (i % 3), b[i])
        for i in range(len(dq)):
            B.add(0, rows[need + i], dq[i])
            B.add(1, rows[need + i], dt[i])
        i = 0
        while len(B.q) < nq or len(B.t) < nt:     # unrelated rows fill what the 1-in-7 gaps left short
            y = rows[(i * 7919) % need] + np.float32(0.125)
            if len(B.q) < nq:
                B.add(0, y, a[(i * 31 + 1) % need])
            if len(B.t) < nt:
                B.add(1, y + np.float32(0.25), b[(i * 37 + 3) % need])
            i += 1
    qd, qy, td, ty = B.finish(nq, nt)
    return qd, qy, td, ty


def band_thresholds(D, qy, ty, max_dy):
    """d* of every query and train: the distance of its mutual band candidate, -1 if it has none."""
    n, m = D.shape
    thq, tht = np.full(n, -1, np.int64), np.full(m, -1, np.int64)
    if n == 0 or m == 0:
        return thq, tht
    band = np.abs(qy[:, None] - ty[None, :]) <= np.float32(max_dy)
    key = np.where(band, D.astype(np.int64) * 65536, np.int64(1) << 40)
    rk = (key + np.arange(m)[None, :]).min(1)
    ck = (key + np.arange(n)[:, None]).min(0)
    for i in range(n):
        if rk[i] < (1 << 40) and ck[rk[i] & 0xFFFF] & 0xFFFF == i:
            thq[i] = rk[i] >> 16
            tht[rk[i] & 0xFFFF] = rk[i] >> 16
    return thq, tht


def test_cross_scenario_covers_every_class_edge():
    """The scenario puts candidate distances on both sides of every split, has entries without a candidate, float32
    |dy| exactly at max_dy, and exact ties across the band edge that the unbanded reference resolves to a lower index."""
    for max_dy in (0.7, 2.0):
        qd, qy, td, ty = cross_scenario(1000, 1000, max_dy, 5)
        assert len(qd) == 1000 and len(td) == 1000
        assert np.all(np.diff(qy) >= 0) and np.all(np.diff(ty) >= 0)
        D = omatch.hamming_matrix(qd, td)
        thq, tht = band_thresholds(D, qy, ty, max_dy)
        assert set(D_STAR) <= set(thq.tolist()), sorted(set(D_STAR) - set(thq.tolist()))
        assert np.any(thq == -1) and np.any(tht == -1)
        dy = np.abs(qy[:, None] - ty[None, :])
        m = np.float32(max_dy)
        assert np.any(dy == m) and np.any((dy > m) & (dy < m + 1e-4)) and np.any((dy < m) & (dy > m - 1e-4))
        has = np.nonzero(thq >= 0)[0]
        row_min, row_arg = D.min(1), D.argmin(1)
        band = np.abs(qy[:, None] - ty[None, :]) <= np.float32(max_dy)
        out_tie = [i for i in has if row_min[i] == thq[i] and not band[i, row_arg[i]]]
        col_min, col_arg = D.min(0), D.argmin(0)
        has_t = np.nonzero(tht >= 0)[0]
        out_tie_c = [j for j in has_t if col_min[j] == tht[j] and not band[col_arg[j], j]]
        assert len(out_tie) >= 10 and len(out_tie_c) >= 10, (len(out_tie), len(out_tie_c))
        # some ties sit exactly on the LB4 / LB8 bound
        tq = np.array(out_tie)
        assert np.any(_lb4(qd[tq], td[row_arg[tq]]) == thq[tq])
        assert np.any((_lb8(qd[tq], td[row_arg[tq]]) == thq[tq]) & (thq[tq] > 24))


# ---- 3. cross-check against the reference -------------------------------------------------------------------------------
def _kps(FE, y, x=None):
    k = np.zeros(len(y), FE.KPOINT)
    k["y"] = y
    k["x"] = 0 if x is None else x
    k["size"] = 31
    return k


def _ref_cross(qd, td, qy, ty, max_dy):
    if max_dy < 0:
        return omatch.cross_check(omatch.hamming_matrix(qd, td))
    return omatch.stereo_match_crosscheck(qy, ty, qd, td, max_dy)


def _assert_same(got, want, what):
    q, t, d = want
    assert len(got) == len(q), (what, len(got), len(q))
    assert np.array_equal(got["queryIdx"], q), what
    assert np.array_equal(got["trainIdx"], t), what
    assert np.array_equal(got["distance"], d.astype(np.float32)), what
    assert np.all(got["imgIdx"] == 0), what


def _run_cross(FE, f, qd, qy, td, ty, max_dy):
    f.profile_reset()
    got = f.stereo_match(_kps(FE, qy), qd, _kps(FE, ty), td, FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE,
                                                                            max_dy=max_dy))
    return got, f.stage_times()["hamming_cross"][1]


SIZES = [(0, 0), (0, 33), (33, 0), (1, 1), (1, 2), (2, 2), (31, 33), (33, 31), (127, 129), (129, 127), (255, 257),
         (257, 255), (2, 1000), (1000, 2), (1000, 1000), (3, 4097), (4097, 3), (4097, 4097)]


@pytest.mark.gpu
@pytest.mark.parametrize("cap", [1000, 16384, 16385])
@pytest.mark.parametrize("max_dy", MAX_DY)
def test_cross_check_paths_vs_reference(FE, cap, max_dy, monkeypatch):
    """Every scenario through the pruned path (with the join up to a capacity of 16384, the LB scan above), the LB scan
    alone (FE_CROSS_MIH=0), the all-pairs kernel (FE_CROSS_PRUNE=0) and without the |dy| filter: bit-exact against the
    oracle, and each call's hamming_cross launch count names the path it took."""
    forms = (("default", None, "join" if cap <= 16384 else "scan"), ("no_mih", "FE_CROSS_MIH", "scan"),
             ("no_prune", "FE_CROSS_PRUNE", "all_pairs"))
    ctx = {}
    try:
        for name, env, _ in forms:
            monkeypatch.delenv("FE_CROSS_MIH", raising=False)
            monkeypatch.delenv("FE_CROSS_PRUNE", raising=False)
            if env:
                monkeypatch.setenv(env, "0")
            ctx[name] = FE.FrontEnd(max_keypoints=cap)
        for i, (nq, nt) in enumerate(s for s in SIZES if max(s) <= cap):
            qd, qy, td, ty = cross_scenario(nq, nt, max_dy, 1000 * i + int(max_dy * 10) + cap)
            want = _ref_cross(qd, td, qy, ty, max_dy)
            for name, _, path in forms:
                got, launches = _run_cross(FE, ctx[name], qd, qy, td, ty, max_dy)
                _assert_same(got, want, (name, nq, nt, max_dy, cap))
                assert launches == CROSS_LAUNCHES[path], (name, nq, nt, launches)
            got, launches = _run_cross(FE, ctx["default"], qd, qy, td, ty, -1.0)
            _assert_same(got, _ref_cross(qd, td, qy, ty, -1.0), ("no filter", nq, nt, cap))
            assert launches == CROSS_LAUNCHES["all_pairs"]
    finally:
        for f in ctx.values():
            f.close()


@pytest.mark.gpu
def test_cross_check_context_reuse_with_changing_sizes(FE):
    """One context, sizes shrinking and growing with different data each call: the scratch arrays (candidates, thresholds,
    permutations, row / column minima, row table) are only partly rewritten, so a stale entry would show here."""
    seq = [(4097, 4097), (3, 2), (1000, 4097), (0, 5), (257, 31), (4097, 1000), (1, 1), (2000, 2000), (33, 4000), (4097, 4097)]
    with FE.FrontEnd(max_keypoints=4200) as f:
        for i, (nq, nt) in enumerate(seq):
            for max_dy in (0.7, 2.0):
                qd, qy, td, ty = cross_scenario(nq, nt, max_dy, 7000 + 13 * i + int(max_dy))
                got, launches = _run_cross(FE, f, qd, qy, td, ty, max_dy)
                _assert_same(got, _ref_cross(qd, td, qy, ty, max_dy), ("reuse", i, nq, nt, max_dy))
                assert launches == CROSS_LAUNCHES["join"]


def _popc32(x):
    x = x - ((x >> 1) & 0x55555555)
    x = (x & 0x33333333) + ((x >> 2) & 0x33333333)
    x = (x + (x >> 4)) & 0x0F0F0F0F
    return ((x * 0x01010101) & 0xFFFFFFFF) >> 24


def key_cross_check(qd, td, qy, ty, max_dy, chunk=256):
    """Cross-check by keys without the N x M matrix: per row and per column the minimum of distance << 16 | index (ties go
    to the lower index, as BFMatcher's first minimum), in chunks with torch integer operations on the GPU."""
    import torch
    dev = torch.device("cuda")
    n, m = len(qd), len(td)
    if n == 0 or m == 0:
        z = np.zeros(0, np.int32)
        return z, z, np.zeros(0, np.float32)
    q = torch.from_numpy(np.ascontiguousarray(qd).view("<u4").astype(np.int64)).to(dev)
    t = torch.from_numpy(np.ascontiguousarray(td).view("<u4").astype(np.int64)).to(dev)
    tidx = torch.arange(m, device=dev, dtype=torch.int64)
    rowkey = torch.empty(n, dtype=torch.int64, device=dev)
    colkey = torch.full((m,), 1 << 40, dtype=torch.int64, device=dev)
    for s in range(0, n, chunk):
        d = _popc32(q[s:s + chunk, None, :] ^ t[None, :, :]).sum(2)
        rowkey[s:s + chunk] = (d * 65536 + tidx[None, :]).min(1).values
        qidx = torch.arange(s, s + d.shape[0], device=dev, dtype=torch.int64)
        colkey = torch.minimum(colkey, (d * 65536 + qidx[:, None]).min(0).values)
    rowkey, colkey = rowkey.cpu().numpy(), colkey.cpu().numpy()
    s = rowkey & 0xFFFF
    qs = np.nonzero((colkey[s] & 0xFFFF) == np.arange(n))[0]
    ts, ds = s[qs], (rowkey[qs] >> 16).astype(np.float32)
    if max_dy >= 0:
        keep = np.abs(qy[qs] - ty[ts]) <= np.float32(max_dy)
        qs, ts, ds = qs[keep], ts[keep], ds[keep]
    return qs.astype(np.int32), ts.astype(np.int32), ds


@pytest.mark.gpu
def test_cross_check_at_full_index_range(FE, monkeypatch):
    """Capacity 65535, the largest fe_create accepts, with up to 65535 entries per side: indices up to 0xFFFE next to the
    padding lanes' 0xFFFF.  The reference is the chunked key cross-check, itself checked against the oracle first."""
    qd, qy, td, ty = cross_scenario(700, 600, 0.7, 3)
    for max_dy in (0.7, -1.0):
        want = _ref_cross(qd, td, qy, ty, max_dy)
        got = key_cross_check(qd, td, qy, ty, max_dy, chunk=64)
        assert all(np.array_equal(a, b) for a, b in zip(got, want))
    cases = [(65535, 41000, 0.7), (40000, 65535, 2.0), (65535, 65535, 0.7)]
    for form, env, path in (("default", None, "scan"), ("no_mih", "FE_CROSS_MIH", "scan"), ("no_prune", "FE_CROSS_PRUNE", "all_pairs")):
        monkeypatch.delenv("FE_CROSS_MIH", raising=False)
        monkeypatch.delenv("FE_CROSS_PRUNE", raising=False)
        if env:
            monkeypatch.setenv(env, "0")
        with FE.FrontEnd(max_keypoints=65535, max_height=16384) as f:      # rows of the scenario's whole y range
            for i, (nq, nt, max_dy) in enumerate(cases if form == "default" else cases[:1]):
                qd, qy, td, ty = cross_scenario(nq, nt, max_dy, 90 + i)
                got, launches = _run_cross(FE, f, qd, qy, td, ty, max_dy)
                _assert_same(got, key_cross_check(qd, td, qy, ty, max_dy), (form, nq, nt, max_dy))
                assert launches == CROSS_LAUNCHES[path], (form, launches)
                if min(nq, nt) > 60000:
                    assert got["queryIdx"].max() > 65000 and got["trainIdx"].max() > 65000
                if form == "default":
                    got, launches = _run_cross(FE, f, qd, qy, td, ty, -1.0)
                    _assert_same(got, key_cross_check(qd, td, qy, ty, -1.0), ("no filter", nq, nt))
                    assert launches == CROSS_LAUNCHES["all_pairs"]


# ---- 4. tuning knobs (read once per process: one subprocess each) --------------------------------------------------------
KNOBS = [{"FE_CX_SWAP": "0"}, {"FE_CX_T": "0", "FE_CX_T2": "0"}, {"FE_CX_T": "64", "FE_CX_T2": "256"},
         {"FE_CX_WIDE": "0", "FE_CX_OVERLAP": "0"}, {"FE_CROSS_MIH": "0", "FE_VERIFY_VARIANT": "2"}]


def knob_scenarios():
    """The fixed set the knob runs check: cross-check scenarios at a capacity with the join and one without, both pair
    counts of the batched pipeline on tiled images.  Raises AssertionError on the first difference from the oracle."""
    import front_end_b200 as FE
    for cap, sizes in ((4200, [(1000, 1000), (3, 4097), (4097, 3), (257, 255)]), (16385, [(4097, 4097)])):
        with FE.FrontEnd(max_keypoints=cap) as f:
            for i, (nq, nt) in enumerate(sizes):
                for max_dy in (0.7, 2.0):
                    qd, qy, td, ty = cross_scenario(nq, nt, max_dy, 300 + i)
                    got, launches = _run_cross(FE, f, qd, qy, td, ty, max_dy)
                    _assert_same(got, _ref_cross(qd, td, qy, ty, max_dy), (cap, nq, nt, max_dy))
                    assert launches in (CROSS_LAUNCHES["join"], CROSS_LAUNCHES["scan"])
    for P in (3, 9):
        _pipeline_vs_oracle(FE, P, seed=500 + P)


@pytest.mark.gpu
@pytest.mark.parametrize("knobs", KNOBS, ids=lambda k: ",".join("%s=%s" % kv for kv in k.items()))
def test_tuning_knobs_are_exact(knobs, tmp_path):
    script = tmp_path / "knobs.py"
    script.write_text("import sys\nsys.path.insert(0, %r)\nsys.path.insert(0, %r)\n"
                      "from test_hamming_exhaustive import knob_scenarios\nknob_scenarios()\nprint('ok')\n"
                      % (ROOT_DIR, os.path.join(ROOT_DIR, "tests")))
    env = {k: v for k, v in os.environ.items() if not k.startswith(("FE_CX_", "FE_CROSS_", "FE_VERIFY_"))}
    env.update(knobs)
    p = subprocess.run([sys.executable, str(script)], env=env, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0 and p.stdout.strip().endswith("ok"), p.stderr[-3000:]


# ---- 5. the batched pipeline on engineered images ------------------------------------------------------------------------
def _box(a, r):
    """Mean over a (2r + 1)^2 box, edges replicated."""
    p = np.pad(a.astype(np.float64), r, mode="edge")
    c = np.cumsum(np.cumsum(p, 0), 1)
    c = np.pad(c, ((1, 0), (1, 0)))
    k = 2 * r + 1
    return (c[k:, k:] - c[:-k, k:] - c[k:, :-k] + c[:-k, :-k]) / (k * k)


def engineered_pair(h, w, seed, disp=12):
    """u8 stereo pair: aperiodic texture plus rectangles that tile one random patch at a period of 40 .. 64 px in x and
    y.  The right image is the left one shifted by `disp` px, so a tiled corner has exact duplicate descriptors in its
    own row (in-band ties) and a period above (out-of-band ties at a lower index)."""
    rng = np.random.default_rng(seed)
    canvas = _box(rng.integers(0, 256, (h, w + disp)), 2) * 0.6 + 50
    for _ in range(4):
        px, py = (int(v) for v in rng.integers(40, 65, 2))
        patch = _box(rng.integers(0, 256, (py, px)), 1)
        nx, ny = int(rng.integers(3, 6)), int(rng.integers(3, 5))
        x0 = int(rng.integers(0, max(1, w + disp - nx * px)))
        y0 = int(rng.integers(0, max(1, h - ny * py)))
        tile = np.tile(patch, (ny, nx))[:h - y0, :w + disp - x0]
        canvas[y0:y0 + tile.shape[0], x0:x0 + tile.shape[1]] = tile
    canvas = np.clip(np.rint(canvas), 0, 255).astype(np.uint8)
    return np.ascontiguousarray(canvas[:, disp:]), np.ascontiguousarray(canvas[:, :w])


def _pipeline_vs_oracle(FE, P, seed, h=480, w=640, n_features=3000):
    """pipeline_batch (mode A band 2.0 ratio 0.8, mode B max_dy 0.7) on P engineered pairs: every pair's match lists equal
    the oracle's on the pipeline's own keypoints and descriptors.  Returns the duplicate counts (in band, out of band)."""
    pairs = [engineered_pair(h, w, seed + p) for p in range(P)]
    Ls, Rs = np.stack([a for a, _ in pairs]), np.stack([b for _, b in pairs])
    cap = 8192
    with FE.FrontEnd(max_width=w, max_height=h, max_pairs=P, max_keypoints=cap, n_features=n_features) as f:
        f.profile_reset()
        out = f.pipeline_batch(Ls, Rs, FE.match_cfg(epi_threshold=2.0, ratio=0.8),
                               FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, max_dy=0.7))
        launches = f.stage_times()["hamming_cross"][1]
    assert launches == CROSS_LAUNCHES["fused_scan" if os.environ.get("FE_CROSS_MIH") == "0" else "fused_join"]
    dup_in = dup_out = 0
    for p in range(P):
        nl, nr = out["n_kps"][2 * p], out["n_kps"][2 * p + 1]
        lk, rk = out["kps"][2 * p][:nl], out["kps"][2 * p + 1][:nr]
        ld, rd = out["desc"][2 * p][:nl], out["desc"][2 * p + 1][:nr]
        q, t, d = omatch.stereo_match_ratio(lk["y"], rk["y"], ld, rd, 2.0, 0.8)
        _assert_same(out["matches_a"][p][:out["n_a"][p]], (q, t, d), ("mode A", P, p))
        q, t, d = omatch.stereo_match_crosscheck(lk["y"], rk["y"], ld, rd, 0.7)
        _assert_same(out["matches_b"][p][:out["n_b"][p]], (q, t, d), ("mode B", P, p))
        D = omatch.hamming_matrix(ld, rd)
        zero = D == 0
        band = np.abs(lk["y"][:, None] - rk["y"][None, :]) <= np.float32(0.7)
        dup_in += int(((zero & band).sum(1) >= 2).sum())                    # queries with two identical trains in band
        dup_out += int(((zero & ~band).any(1) & (zero & band).any(1)).sum())   # ... and one out of band as well
    return dup_in, dup_out


@pytest.mark.gpu
@pytest.mark.parametrize("P", [9, 3])
def test_pipeline_on_tiled_images_vs_oracle(FE, P):
    """Fused band (mode A's kNN-2 also yields mode B's candidates), the wide-band kill of false candidates and the fused
    ratio finalize, on images whose tiled regions produce exact duplicate descriptors in band and out of band."""
    dup_in, dup_out = _pipeline_vs_oracle(FE, P, seed=40 + P)
    assert dup_in >= 20 * P and dup_out >= 20 * P, (dup_in, dup_out)


# ---- 6. kNN-2 and the ratio test ----------------------------------------------------------------------------------------
RATIO_PAIRS = ((8, 10), (3, 4), (0, 0), (0, 1), (4, 5), (12, 15), (16, 20), (24, 30), (9, 12), (7, 9), (10, 10), (1, 2))


def knn_scenario(seed, thr, h2=False):
    """Raster-ordered queries and trains: per query a best train at d0 and a second at d1 (RATIO_PAIRS, ratios exact in
    double), a tie for the second at a higher index, a tie for the best just outside the band (lower index) and at
    exactly |dy| == thr, singleton rows, rows without a train, and unrelated background."""
    rng = np.random.default_rng(seed)
    m = np.float32(thr)
    B = _Builder()
    Y = np.float32(0.5)
    if thr > 0:                                         # |dy| == thr exactly in float32 needs rows near y = 0
        q = rng.integers(0, 256, 32, dtype=np.uint8)
        B.add(0, m, q)
        B.add(1, 0.0, _flip(q, bits_hamming2(8, rng) if h2 else bits_tight_lb4(8, rng)))
        B.add(1, 0.0, _flip(q, bits_hamming2(10, rng) if h2 else bits_tight_lb4(10, rng)))
        Y = np.float32(m + 1)
    for i in range(240):
        d0, d1 = RATIO_PAIRS[i % len(RATIO_PAIRS)]
        q = rng.integers(0, 256, 32, dtype=np.uint8)

        def near(k):
            return _flip(q, bits_hamming2(k, rng) if h2 else BITS["tight4" if k <= 32 else "random"][0](k, rng))

        qy = Y + np.float32(2 * m + 3)
        yp = _y_pair(qy, m, 0) if i % 3 == 0 else None
        ty = yp[1] if yp is not None else qy
        if yp is not None and i % 2:
            ty = np.float32(2 * qy - ty)                # the train below the query instead of above
        B.add(0, qy, q)
        kind = i % 6
        if kind != 5:
            B.add(1, ty, near(d0))
        if kind in (0, 1, 2, 3):
            B.add(1, ty, near(d1))
        if kind in (1, 3):
            B.add(1, ty, near(d1))                      # a tie for the second place, higher index
        if kind in (2, 3):
            B.add(1, Y, near(d0))                       # a tie for the best outside the band, lower index
        if kind == 4:
            B.add(0, qy, near(d0 + 1))                  # a second query of the row
        Y = np.float32(qy + 2 * m + 3)
    a, b = unrelated(300, 300, rng)
    ys = Y + np.sort(rng.integers(0, 120, 300)).astype(np.float32) * np.float32(0.5)
    for i in range(300):
        B.add(0, ys[i], a[i])
        B.add(1, ys[(i * 7) % 300], b[i])
    return B.finish(10 ** 9, 10 ** 9)


@pytest.mark.gpu
@pytest.mark.parametrize("h2", [False, True])
@pytest.mark.parametrize("thr", [0.0, 0.7, 2.0])
def test_knn2_band_and_general_kernels(FE, h2, thr):
    """Masked kNN-2 through the band kernel (raster-ordered trains) and the general kernel (the same trains shuffled), with
    NORM_HAMMING and NORM_HAMMING2, and unmasked: (best, second) indices and distances equal the oracle's, ties included."""
    qd, qy, td, ty = knn_scenario(11 + int(10 * thr), thr, h2)
    norm = FE.NORM_HAMMING2 if h2 else FE.NORM_HAMMING
    D = (omatch.hamming2_matrix if h2 else omatch.hamming_matrix)(qd, td)
    perm = np.random.default_rng(1).permutation(len(td))
    with FE.FrontEnd(max_keypoints=4096) as f:
        for order in (np.arange(len(td)), perm):
            tdo, tyo = td[order], ty[order]
            Do = D[:, order]
            cfg = FE.match_cfg(mask=FE.MASK_EPIPOLAR, epi_threshold=thr, norm=norm)
            f.profile_reset()
            idx, dist = f.knnMatch(_kps(FE, qy), qd, _kps(FE, tyo), tdo, cfg)
            assert f.stage_times()["hamming_knn2"][1] == (2 if order is not perm else 1)
            oi, od, _ = omatch.knn2(Do, omatch.epipolar_mask(qy, tyo, thr))
            assert np.array_equal(idx, oi) and np.array_equal(dist, od), (thr, h2, order is perm)
            idx, dist = f.knnMatch(_kps(FE, qy), qd, _kps(FE, tyo), tdo, FE.match_cfg(mask=FE.MASK_NONE, norm=norm))
            oi, od, _ = omatch.knn2(Do)
            assert np.array_equal(idx, oi) and np.array_equal(dist, od)
        # the band has exact boundary rows and second-place ties
        assert np.any(np.abs(qy[:, None] - ty[None, :]) == np.float32(thr))


@pytest.mark.gpu
@pytest.mark.parametrize("h2", [False, True])
def test_knn2_window_list_flushes(FE, h2):
    """The window variant compacts the trains that pass |dx| < w/2 into a per-warp list of 256 and measures it whenever it
    fills: 1500 trains inside one query's box flush it several times; the box edges are hit exactly."""
    rng = np.random.default_rng(8)
    nq, nt = 200, 1500
    qd = rng.integers(0, 256, (nq, 32), dtype=np.uint8)
    td = rng.integers(0, 256, (nt, 32), dtype=np.uint8)
    td[::5] = qd[rng.integers(0, nq, len(td[::5]))]                    # exact duplicates: ties for best and second
    td[1::5] = [_flip(qd[i], bits_tight_lb4(3, rng)) for i in rng.integers(0, nq, len(td[1::5]))]
    qy = np.sort(rng.uniform(100, 140, nq)).astype(np.float32)
    ty = np.sort(np.concatenate([rng.uniform(95, 145, nt - 100), np.full(50, 100.0), np.full(50, 170.0)])).astype(np.float32)
    qx = rng.uniform(400, 440, nq).astype(np.float32)
    tx = rng.uniform(360, 480, nt).astype(np.float32)
    tx[:40] = qx[0] + 50.0                                              # |dx| == w/2 exactly: outside the box
    tx[40:80] = qx[1] - 49.0
    norm = FE.NORM_HAMMING2 if h2 else FE.NORM_HAMMING
    D = (omatch.hamming2_matrix if h2 else omatch.hamming_matrix)(qd, td)
    with FE.FrontEnd(max_keypoints=2048) as f:
        for ww, wh in ((100, 100), (100, 60), (1000, 200)):
            idx, dist = f.knnMatch(_kps(FE, qy, qx), qd, _kps(FE, ty, tx), td, FE.match_cfg(mask=FE.MASK_WINDOW, win_w=ww, win_h=wh,
                                                                                             norm=norm))
            mask = omatch.window_mask(qx, qy, tx, ty, ww, wh)
            oi, od, _ = omatch.knn2(D, mask)
            assert np.array_equal(idx, oi) and np.array_equal(dist, od), (ww, wh)
            if ww == 1000:
                assert mask.sum(1).max() > 4 * 256


@pytest.mark.gpu
@pytest.mark.parametrize("ratio", [0.8, 0.75, 1.0, 0.0])
def test_ratio_boundaries(FE, ratio):
    """Lowe's test is d0 < ratio * d1 in double, strict: 8 / 10 at 0.8 and 3 / 4 at 0.75 are rejected, 0 / 0 is rejected,
    a singleton row is accepted, ratio 1.0 keeps only strict improvements and ratio 0.0 only singletons."""
    qd, qy, td, ty = knn_scenario(21, 2.0)
    cfg = FE.match_cfg(mask=FE.MASK_EPIPOLAR, epi_threshold=2.0, ratio=ratio)
    D = omatch.hamming_matrix(qd, td)
    oi, od, cnt = omatch.knn2(D, omatch.epipolar_mask(qy, ty, 2.0))
    want = omatch.lowe_ratio(oi, od, ratio)
    with FE.FrontEnd(max_keypoints=4096) as f:
        got = f.stereo_match(_kps(FE, qy), qd, _kps(FE, ty), td, cfg)
    _assert_same(got, want, ratio)
    exact = (cnt == 2) & (od[:, 0].astype(np.float64) == ratio * od[:, 1].astype(np.float64))
    assert np.any(cnt == 1) and np.any((cnt == 2) & (od[:, 0] == 0) & (od[:, 1] == 0))
    if ratio in (0.8, 0.75, 1.0):
        assert np.any(exact & (od[:, 0] > 0))                        # rows exactly on the boundary, rejected
    want_pipe = omatch.stereo_match_ratio(qy, ty, qd, td, 2.0, ratio)
    assert all(np.array_equal(a, b) for a, b in zip(want, want_pipe))
