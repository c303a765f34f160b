"""Ranking comparators for the parity tests.

Contract (BASELINE.json north_star): returned ids and rank order are bit-exact except where
scores fall within a stated relative tolerance of a tie.  ``assert_same_ranking`` implements
exactly that: positions whose reference scores are within ``rel_tol`` of each other form a tie
cluster; within a cluster any order is accepted; the last cluster may exchange members with
items that fell just below the cut-off (they are checked by score instead).

The sparse branch is bit-exact, so it is held to more: ``assert_same_list`` requires the very same
(row, score) sequence, scores equal bit for bit — the total order (score desc, row asc) decides
every tie, including the ones at the k'-th position.
"""
from __future__ import annotations

import struct


def _bits(x) -> bytes:
    return struct.pack("<d", float(x))


def assert_same_list(got, want, what=""):
    """got / want: sequences of (row, score).  Identical rows in identical order, scores bit-equal."""
    got = [(int(g[0]), float(g[1])) for g in got]
    want = [(int(w[0]), float(w[1])) for w in want]
    for i, (g, w) in enumerate(zip(got, want)):
        assert g[0] == w[0] and _bits(g[1]) == _bits(w[1]), \
            f"{what}: rank {i}: got {g} want {w}\n got={got[max(0, i - 3):i + 4]}\nwant={want[max(0, i - 3):i + 4]}"
    assert len(got) == len(want), f"{what}: length {len(got)} != {len(want)}\n got={got[-4:]}\nwant={want[-4:]}"


def _close(a: float, b: float, rel_tol: float, abs_tol: float) -> bool:
    return abs(a - b) <= max(abs_tol, rel_tol * max(abs(a), abs(b)))


def assert_same_ranking(got, want, rel_tol=0.0, abs_tol=0.0, what=""):
    """got / want: sequences of (label, score).  Scores must agree position by position
    within tolerance; labels must agree up to permutation inside tie clusters."""
    got = [(g[0], float(g[1])) for g in got]
    want = [(w[0], float(w[1])) for w in want]
    assert len(got) == len(want), f"{what}: length {len(got)} != {len(want)}\n got={got}\nwant={want}"
    for i, (g, w) in enumerate(zip(got, want)):
        assert _close(g[1], w[1], rel_tol, abs_tol), \
            f"{what}: score mismatch at rank {i}: got {g} want {w}"
    i, n = 0, len(want)
    while i < n:
        j = i + 1
        while j < n and _close(want[j][1], want[j - 1][1], rel_tol, abs_tol):
            j += 1
        gl = sorted(str(x[0]) for x in got[i:j])
        wl = sorted(str(x[0]) for x in want[i:j])
        if gl != wl:
            # only the final cluster may trade members with just-below-cut-off ties
            assert j == n, f"{what}: ids differ in ranks [{i},{j}): got {got[i:j]} want {want[i:j]}"
        i = j


def assert_topk_valid(got, all_scores, passing, k, rel_tol, abs_tol=0.0, what=""):
    """Size-independent check against a full oracle score vector: ``got`` (label=row, score)
    must be sorted, each score must match the oracle score of its row, every returned row must
    pass the filter, and no excluded passing row may beat the k-th returned score by more than
    the tolerance."""
    import numpy as np

    rows = [int(g[0]) for g in got]
    assert len(set(rows)) == len(rows), f"{what}: duplicate rows"
    elig = np.flatnonzero(passing & np.isfinite(all_scores))
    assert len(got) == min(k, len(elig)), f"{what}: got {len(got)} results, expected {min(k, len(elig))}"
    for i, (r, s) in enumerate(got):
        assert passing[int(r)], f"{what}: row {r} does not pass the filter"
        assert _close(float(s), float(all_scores[int(r)]), rel_tol, abs_tol), \
            f"{what}: rank {i} row {r}: score {s} vs oracle {all_scores[int(r)]}"
        if i:
            assert float(got[i - 1][1]) >= float(s) or _close(float(got[i - 1][1]), float(s), rel_tol, abs_tol), \
                f"{what}: not sorted at rank {i}"
    if len(got) and len(elig) > len(got):
        kth = min(float(all_scores[r]) for r in rows)
        rest = np.setdiff1d(elig, np.array(rows, dtype=elig.dtype))
        best_out = float(all_scores[rest].max())
        assert best_out <= kth or _close(best_out, kth, rel_tol, abs_tol), \
            f"{what}: excluded row scores {best_out} > k-th returned {kth}"
