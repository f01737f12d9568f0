"""Descriptors that sit on the edges of the pruned cross-check's multi-index join for 128-bit rows (BRIEF-16).

BRIEF-16 rows ride zero-padded in the 256-bit rows, so launch_hamming_cross_pruned (match.cu) joins on the 8 data halves only
and ends class A at 7 differing bits: at most 7 differing bits leave one of 8 halves identical.  The band pass resolves every
pair inside the |dy| band exactly, so the join only matters for a close partner OUTSIDE the band that beats an entry's mutual
band candidate.  join128_scenario plants exactly those: for a band pair (q0, t0) at d = 7 (one identical data half) or
d = 8 (none), a train that ties with t0 for q0 at a lower index, or beats it at d - 1, on an earlier row outside the band;
and the same on the column side (a query for t0).  The disturbers are class-A entries themselves (a close partner of
their own, or none), so at d = 7 only the join can find them, and at d = 8 only the class-B scans can: a class-A bound of 8
would move those pairs into the join, where no identical half exists.  These CPU tests check that the generator does what
it says; tests/test_batch_brief.py runs the scenario through fe_stereo_match on the GPU.
"""
import numpy as np

from oracle import match as omatch

MAX_DY = 0.7
ROW = 3.0                # rows of one group are this far apart: more than MAX_DY


def flip(row, bits):
    r = row.copy()
    for b in np.asarray(bits, np.int64):
        r[b // 8] ^= np.uint8(1 << int(b % 8))
    return r


def spread(k, rng):
    """k <= 8 bits of a 128-bit row, one in each of k distinct 16-bit halves: k = 7 leaves exactly one half identical, 8 none."""
    return 16 * rng.choice(8, k, replace=False) + rng.integers(0, 16, k)


# what disturbs the band pair (q0, t0) of a group, from a row before the band (lower indices) or after it
KINDS = ("row_tie", "col_tie", "row_closer", "col_closer", "row_tie_after", "none")


def join128_scenario(nq, nt, seed):
    """(qd, qy, td, ty): raster-ordered 16-byte rows built from planted groups (see the module docstring) and, every
    seventh group, unrelated rows."""
    rng = np.random.default_rng(seed)
    q, t = [], []
    g = 0
    while len(q) < nq or len(t) < nt:
        y_out, y0, y_after = (np.float32(ROW * (3 * g + i)) for i in range(3))
        if g % 7 == 6:
            q.append((y0, len(q), rng.integers(0, 256, 16, dtype=np.uint8)))
            t.append((y0, len(t), rng.integers(0, 256, 16, dtype=np.uint8)))
            g += 1
            continue
        d = 7 if g % 2 == 0 else 8
        kind = KINDS[(g // 2) % len(KINDS)]
        partner = (g // (2 * len(KINDS))) % 2 == 1            # the disturber's own close partner on its row, or none
        q0 = rng.integers(0, 256, 16, dtype=np.uint8)
        t0 = flip(q0, spread(d, rng))
        q.append((y0, len(q), q0))
        t.append((y0, len(t), t0))
        k = d if kind.endswith("tie") or kind == "row_tie_after" else d - 1
        if kind.startswith("row"):
            c = flip(q0, spread(k, rng))
            yc = y_after if kind == "row_tie_after" else y_out
            t.append((yc, len(t), c))
            if partner:
                q.append((yc, len(q), flip(c, spread(3, rng))))
        elif kind.startswith("col"):
            c = flip(t0, spread(k, rng))
            q.append((y_out, len(q), c))
            if partner:
                t.append((y_out, len(t), flip(c, spread(3, rng))))
        g += 1
    out = []
    for lst, n in ((q, nq), (t, nt)):
        lst = sorted(lst, key=lambda e: (e[0], e[1]))[:n]
        out += [np.stack([e[2] for e in lst]) if lst else np.zeros((0, 16), np.uint8),
                np.array([e[0] for e in lst], np.float32)]
    return out


def band_candidates(D, qy, ty):
    """Mutual row / column arg-mins inside the |dy| band: (q, t, d*) of every candidate, and every entry's d* (-1: none)."""
    band = np.abs(qy[:, None] - ty[None, :]) <= np.float32(MAX_DY)
    Db = np.where(band, D.astype(np.int64), 1 << 20)
    rq = np.argmin(Db, 1) if D.shape[1] else np.zeros(0, np.int64)
    ct = np.argmin(Db, 0) if D.shape[0] else np.zeros(0, np.int64)
    qs = [i for i in range(D.shape[0]) if Db[i, rq[i]] < (1 << 20) and ct[rq[i]] == i]
    dq, dt = np.full(D.shape[0], -1), np.full(D.shape[1], -1)
    for i in qs:
        dq[i] = dt[rq[i]] = D[i, rq[i]]
    return [(i, int(rq[i]), int(D[i, rq[i]])) for i in qs], dq, dt


def halves_same(a, b):
    return int((a.view("<u2") == b.view("<u2")).sum())


def test_planted_distances_and_halves():
    rng = np.random.default_rng(0)
    for k in range(9):
        row = rng.integers(0, 256, 16, dtype=np.uint8)
        other = flip(row, spread(k, rng))
        assert omatch.hamming_matrix(row[None], other[None])[0, 0] == k
        assert halves_same(row, other) == 8 - k


def test_scenario_plants_out_of_band_disturbers_of_both_classes():
    """Band candidates at d* = 7 and 8 lose their row and their column to class-A entries outside the band; at 7 the winner
    shares exactly one data half with its partner, at 8 none."""
    qd, qy, td, ty = join128_scenario(1200, 1200, 5)
    D = omatch.hamming_matrix(qd, td).astype(np.int64)
    cands, dq, dt = band_candidates(D, qy, ty)
    q_ok, t_ok, _ = omatch.stereo_match_crosscheck(qy, ty, qd, td, MAX_DY)
    kept = set(zip(q_ok.tolist(), t_ok.tolist()))
    seen = {}
    for i, j, d in cands:
        if (i, j) in kept or d > 8:          # (the unrelated background rows lose to anything: d* ~ 64)
            continue
        row_win = int(np.argmin(D[i]))                   # first minimum = BFMatcher's tie rule
        col_win = int(np.argmin(D[:, j]))
        side, win, dist, pair = (("row", row_win, D[i, row_win], (qd[i], td[row_win])) if row_win != j else
                                 ("col", col_win, D[col_win, j], (qd[col_win], td[j])))
        assert win != (j if side == "row" else i)
        outside = abs(float(qy[i] - ty[win])) > MAX_DY if side == "row" else abs(float(qy[win] - ty[j])) > MAX_DY
        assert outside, (i, j, side)                       # the band pass cannot see the winner
        disturber_dstar = dt[win] if side == "row" else dq[win]
        assert disturber_dstar <= 7, (i, j, side, disturber_dstar)     # the winner is a class-A entry
        if dist == d:
            assert halves_same(*pair) == (1 if d == 7 else 0), (i, j, d)
        seen[(d, side, int(dist == d))] = seen.get((d, side, int(dist == d)), 0) + 1
    for d in (7, 8):
        for side in ("row", "col"):
            for tie in (0, 1):
                assert seen.get((d, side, tie), 0) >= 5, (d, side, tie, seen)
    # the controls survive: ties at a HIGHER index outside the band, and undisturbed pairs
    assert len(kept) > 300
    assert any(d == 7 for _, _, d in cands) and any(d == 8 for _, _, d in cands)


def test_scenario_sizes_and_order():
    for n in (0, 1, 257, 4097):
        qd, qy, td, ty = join128_scenario(n, n, n + 3)
        assert qd.shape == (n, 16) and td.shape == (n, 16)
        assert np.all(np.diff(qy) >= 0) and np.all(np.diff(ty) >= 0)
