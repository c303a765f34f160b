"""K3M (posting-driven MaxScore sparse scoring, csrc/sparse_ms.cuh) on the CPU: the host/device functions
that carry the kernel's logic are compiled with g++ (tests/csrc/ms_emul.cpp drives them like the two
kernels do) and every candidate set is compared with the oracle's sparse_dot_product — rows AND fp32
scores bit for bit.  This is the development-container stand-in for the GPU parity tests."""
from __future__ import annotations

import ctypes as C
import math
import subprocess
from pathlib import Path

import numpy as np
import pytest

import _coded
import _data
from oracle import oracle

ROOT = Path(__file__).resolve().parents[1]
SRC = ROOT / "tests" / "csrc" / "ms_emul.cpp"


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    so = tmp_path_factory.mktemp("ms_emul") / "ms_emul.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-o", str(so), str(SRC)],
                   check=True, capture_output=True)
    lib = C.CDLL(str(so))
    vp = C.c_void_p
    lib.ms_emul_segment.restype = C.c_int
    lib.ms_emul_segment.argtypes = ([vp, vp, vp, C.c_uint32, vp, vp, vp, vp, vp, vp, C.c_uint32, vp, vp, vp, vp, vp, vp, vp, C.c_float]
                                    + [C.c_uint32] * 5 + [C.c_uint64, C.c_uint64, vp, vp, C.c_uint32, vp])
    lib.mh_emul_segment.restype = C.c_int
    lib.mh_emul_segment.argtypes = ([vp, vp, vp, C.c_uint32, vp, vp, vp, vp, vp, vp, C.c_uint32, vp, vp, vp, vp, vp, vp, vp, C.c_float]
                                    + [C.c_uint32] * 5 + [vp, vp, C.c_uint32, vp])
    return lib


def _index_of(indptr, terms, vals, corpus=None):
    """Inverted index, dense columns and forward CSR of a corpus, as the library builds them."""
    n = len(indptr) - 1
    rows = np.repeat(np.arange(n, dtype=np.uint32), np.diff(indptr))
    order = np.lexsort((rows, terms))
    post_row, post_val, post_term = rows[order], vals[order], terms[order]
    uniq, start = np.unique(post_term, return_index=True)
    ptr = np.append(start, len(post_term)).astype(np.int64)
    df = np.diff(ptr)
    maxval = np.maximum.reduceat(post_val, start)
    heavy = [i for i in np.argsort(-df) if df[i] * 8 >= n][:64]
    stride = (n + 2 + 63) // 64 * 64
    hv = np.full((max(1, len(heavy)), stride), np.nan, np.float32)
    hof = {}
    for k, i in enumerate(heavy):
        hv[k, post_row[ptr[i]:ptr[i + 1]]] = post_val[ptr[i]:ptr[i + 1]]
        hof[int(uniq[i])] = k
    tab_off, tab_shift, tabs, total = {}, {}, [], 0
    for i in range(len(uniq)):                       # bucket tables, as ensure_sparse_index builds them
        d = int(df[i])
        if d < 32:
            continue
        shift = 0
        while shift < 31 and (d << (shift + 1)) <= n * 4:
            shift += 1
        if i in heavy:
            shift = max(shift, 12)
        nb = (n >> shift) + 2
        targets = np.arange(nb, dtype=np.int64) << shift
        tabs.append((np.searchsorted(post_row[ptr[i]:ptr[i + 1]], targets, side="left") + ptr[i]).astype(np.uint32))
        tab_off[int(uniq[i])], tab_shift[int(uniq[i])] = total, shift
        total += nb
    term_tab = np.concatenate(tabs) if tabs else np.zeros(1, np.uint32)
    return dict(term_tab=term_tab, tab_off=tab_off, tab_shift=tab_shift, corpus=corpus, n=n, indptr=indptr, terms=terms, vals=vals, post_row=np.ascontiguousarray(post_row),
                post_val=np.ascontiguousarray(post_val), uniq=uniq, ptr=ptr, df=df, maxval=maxval, hv=hv, stride=stride, hof=hof)


@pytest.fixture(scope="module")
def index():
    """A small BM25-style corpus: random document lengths, so exact score ties are rare."""
    corpus = _data.make_corpus(seed=11, n=9000, dim=8, vocab=300)
    coded = _coded.code_corpus(corpus)
    return _index_of(*coded["csr"], corpus=corpus)


TIE_A, TIE_B = 1000, 2000


@pytest.fixture(scope="module")
def ties_index():
    """A corpus where most scores tie: term A on the odd rows, term B on the even rows (equal df, so a query [A, B]
    weighs them equally), values from {0.5, 0.75, 1.0, 1.25}, one extra non-query term per row, and every 37th row
    with a query-term value of 0.0 (score 0, still a candidate: it overlaps the query).  The postings of A and B
    interleave in row order, so a stage that walks them in position order meets tied rows out of row order."""
    n = 6000
    rng = np.random.RandomState(17)
    val = rng.choice(np.float32([0.5, 0.75, 1.0, 1.25]), size=n)
    val[::37] = 0.0
    extra = 3000 + rng.randint(0, 50, size=n)
    indptr = np.arange(0, 2 * n + 1, 2, dtype=np.int64)
    terms = np.empty(2 * n, np.uint32)
    vals = np.empty(2 * n, np.float32)
    terms[0::2] = np.where(np.arange(n) % 2 == 1, TIE_A, TIE_B)
    vals[0::2] = val
    terms[1::2] = extra
    vals[1::2] = rng.choice(np.float32([0.5, 1.0]), size=n)
    return _index_of(indptr, terms, vals)


def _tie_query(ix, extra_term=None):
    """[A, B] (plus optionally one extra term) with the IDF weights of the index: A and B weigh exactly the same."""
    n = ix["n"]
    dfm = {int(t): int(d) for t, d in zip(ix["uniq"], ix["df"])}
    q_idx = sorted([TIE_A, TIE_B] + ([extra_term] if extra_term is not None else []))
    return q_idx, [math.log((n - dfm[t] + 0.5) / (dfm[t] + 0.5) + 1.0) for t in q_idx]


def _reference(ix, q_idx, q_w, r0, r1, mask_bits, tau):
    out = {}
    for r in range(r0, r1):
        if mask_bits is not None and not (mask_bits[r >> 5] >> (r & 31)) & 1:
            continue
        a, b = ix["indptr"][r], ix["indptr"][r + 1]
        s = oracle.sparse_dot_product(q_idx, q_w, ix["terms"][a:b].tolist(), [float(x) for x in ix["vals"][a:b]])
        if s is not None and np.float32(s) >= np.float32(tau):
            out[r] = np.float32(s)
    return out


def _run(emul, ix, q_idx, q_w, r0, r1, mask_bits, tau, chunk, budget, use_tabs=True, use_heavy=True, stage=(0, 2 ** 63), mh_max_post=None):
    nt = len(q_idx)
    qt = np.asarray(q_idx, np.uint32)
    qw = np.asarray(q_w, np.float64)
    slot = np.searchsorted(ix["uniq"], qt)
    ok = (slot < len(ix["uniq"])) & (ix["uniq"][np.minimum(slot, len(ix["uniq"]) - 1)] == qt)
    plo = np.where(ok, ix["ptr"][np.minimum(slot, len(ix["uniq"]) - 1)], 0).astype(np.uint32)
    phi = np.where(ok, ix["ptr"][np.minimum(slot, len(ix["uniq"]) - 1) + 1], 0).astype(np.uint32)
    ub = np.where(ok, qw * ix["maxval"][np.minimum(slot, len(ix["uniq"]) - 1)].astype(np.float64), 0.0)
    hidx = np.asarray([ix["hof"].get(int(t), -1) if use_heavy else -1 for t in qt], np.int32)
    qtab = np.asarray([ix["tab_off"].get(int(t), 0xFFFFFFFF) if use_tabs else 0xFFFFFFFF for t in qt], np.uint32)
    qshift = np.asarray([ix["tab_shift"].get(int(t), 0) for t in qt], np.uint8)
    cap = ix["n"] + 8
    out_rows = np.zeros(cap, np.uint32)
    out_scores = np.zeros(cap, np.float32)
    stats = np.zeros(4, np.uint64)
    p = lambda a: None if a is None else C.c_void_p(a.ctypes.data)
    if mh_max_post is not None:             # K3H: hash-accumulate per row range
        rc = emul.mh_emul_segment(p(ix["post_row"]), p(ix["post_val"]), p(ix["hv"]), ix["stride"], p(ix["term_tab"]), p(qtab), p(qshift),
                                  p(ix["indptr"]), p(ix["terms"]),
                                  p(ix["vals"]), nt, p(qt), p(qw), p(ub), p(hidx), p(plo), p(phi), p(mask_bits), C.c_float(tau),
                                  r0, r1, ix["n"], budget, mh_max_post, p(out_rows), p(out_scores), cap, p(stats))
    else:
        rc = emul.ms_emul_segment(p(ix["post_row"]), p(ix["post_val"]), p(ix["hv"]), ix["stride"], p(ix["term_tab"]), p(qtab), p(qshift),
                                  p(ix["indptr"]), p(ix["terms"]),
                                  p(ix["vals"]), nt, p(qt), p(qw), p(ub), p(hidx), p(plo), p(phi), p(mask_bits), C.c_float(tau),
                                  r0, r1, ix["n"], chunk, budget, stage[0], stage[1], p(out_rows), p(out_scores), cap, p(stats))
    assert rc >= 0, f"emulation failed rc={rc}"
    got = {}
    for r, s in zip(out_rows[:rc], out_scores[:rc]):
        assert int(r) not in got, f"row {r} reported twice (ownership broken)"
        got[int(r)] = np.float32(s)
    return got, stats


def _query(ix, seed, nnz):
    corpus = ix["corpus"]
    (_, (idx, val)), = _data.make_queries(seed, corpus, 1, nnz=nnz)
    q_idx, q_val = oracle._sort_sparse(idx, val)
    n = ix["n"]
    dfm = {int(t): int(d) for t, d in zip(ix["uniq"], ix["df"])}
    w = [float(v) * math.log((n - dfm.get(t, 0) + 0.5) / (dfm.get(t, 0) + 0.5) + 1.0) for t, v in zip(q_idx, q_val)]
    return q_idx, w


def _check_candidates(emul, ix, q_idx, w, mask_bits):
    """Every threshold, segment, chunk, budget and lookup kind: the candidates are the rows whose score reaches tau (a
    row that equals tau may still win its tie on the row id), with the oracle's score bits."""
    n = ix["n"]
    full = _reference(ix, q_idx, w, 0, n, mask_bits, -np.inf)
    ranked = sorted(full.values(), reverse=True)
    taus = [-np.inf, 0.0, float(ranked[min(len(ranked) - 1, 30)]), float(ranked[min(len(ranked) - 1, 300)]), float(ranked[0])]
    for tau in taus:
        for (r0, r1) in ((0, n), (2048, n), (2048, 6144)):
            want = {r: s for r, s in full.items() if r0 <= r < r1 and s >= np.float32(tau)}
            for chunk, budget, tabs, heavy in ((512, 100, True, True), (2048, 20, False, True), (512, 100, True, False)):
                got, stats = _run(emul, ix, q_idx, w, r0, r1, mask_bits, np.float32(tau), chunk, budget, tabs, heavy)
                assert got.keys() == want.keys(), (tau, r0, r1, chunk, sorted(set(got) ^ set(want))[:10])
                bad = [r for r in want if got[r].tobytes() != want[r].tobytes()]
                assert not bad, f"score bits differ for rows {bad[:5]}"


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("masked", [False, True])
def test_candidates_match_oracle(emul, index, seed, masked):
    ix = index
    q_idx, w = _query(ix, 100 + seed, (3, 12) if seed % 2 == 0 else (10, 40))
    rng = np.random.RandomState(seed)
    mask_bits = rng.randint(0, 2 ** 32, size=(ix["n"] + 31) // 32, dtype=np.uint64).astype(np.uint32) if masked else None
    _check_candidates(emul, ix, q_idx, w, mask_bits)


@pytest.mark.parametrize("extra", [None, 3007])
@pytest.mark.parametrize("masked", [False, True])
def test_candidates_match_oracle_on_ties(emul, ties_index, extra, masked):
    ix = ties_index
    q_idx, w = _tie_query(ix, extra)
    assert w[q_idx.index(TIE_A)] == w[q_idx.index(TIE_B)]
    rng = np.random.RandomState(3)
    mask_bits = rng.randint(0, 2 ** 32, size=(ix["n"] + 31) // 32, dtype=np.uint64).astype(np.uint32) if masked else None
    _check_candidates(emul, ix, q_idx, w, mask_bits)


def test_pruning_skips_most_postings(emul, index):
    """With an established threshold only a small part of the posting mass is essential."""
    ix = index
    n = ix["n"]
    tot_all = tot_ess = 0
    for seed in range(8):
        q_idx, w = _query(ix, 300 + seed, (3, 12))
        full = _reference(ix, q_idx, w, 0, 2048, None, -np.inf)
        ranked = sorted(full.values(), reverse=True)
        tau = float(ranked[min(len(ranked) - 1, 29)])
        _, stats = _run(emul, ix, q_idx, w, 2048, n, None, np.float32(tau), 512, 100)
        dfm = {int(t): int(d) for t, d in zip(ix["uniq"], ix["df"])}
        tot_all += sum(dfm.get(t, 0) for t in q_idx) * (n - 2048) / n
        tot_ess += int(stats[0])
    assert tot_ess < 0.5 * tot_all, (tot_ess, tot_all)


def test_stress_values(emul, index):
    """Denormal / huge / zero posting values and weights: the order-free sum must still round to the
    reference's fp32 score or fall back to the exact re-score."""
    ix = dict(index)
    rng = np.random.RandomState(5)
    vals = ix["vals"].copy()
    pick = rng.rand(len(vals))
    vals[pick < 0.05] = 0.0
    vals[(pick >= 0.05) & (pick < 0.10)] = np.float32(1e-40)
    vals[(pick >= 0.10) & (pick < 0.15)] = np.float32(3e30)
    vals[(pick >= 0.15) & (pick < 0.30)] *= np.float32(1.0 + 2 ** -20)
    n = ix["n"]
    indptr, terms = ix["indptr"], ix["terms"]
    rows = np.repeat(np.arange(n, dtype=np.uint32), np.diff(indptr))
    order = np.lexsort((rows, terms))
    ix["vals"] = vals
    ix["post_val"] = np.ascontiguousarray(vals[order])
    start = ix["ptr"][:-1]
    ix["maxval"] = np.maximum.reduceat(ix["post_val"], start)
    hv = np.full_like(ix["hv"], np.nan)
    for t, k in ix["hof"].items():
        i = int(np.searchsorted(ix["uniq"], t))
        hv[k, ix["post_row"][ix["ptr"][i]:ix["ptr"][i + 1]]] = ix["post_val"][ix["ptr"][i]:ix["ptr"][i + 1]]
    ix["hv"] = hv
    for seed in range(4):
        q_idx, w = _query(ix, 500 + seed, (8, 30))
        w = [x * (1.0 + 1e-3 * k) for k, x in enumerate(w)]
        full = _reference(ix, q_idx, w, 0, n, None, -np.inf)
        ranked = sorted(full.values(), reverse=True)
        for tau in (-np.inf, float(ranked[min(len(ranked) - 1, 50)])):
            want = {r: s for r, s in full.items() if s >= np.float32(tau)}
            got, _ = _run(emul, ix, q_idx, w, 0, n, None, np.float32(tau), 512, 100)
            assert got.keys() == want.keys()
            assert all(got[r].tobytes() == want[r].tobytes() for r in want)


def _check_stages(emul, ix, q_idx, w, mask_bits, ks, first=16):
    """The staged flow of a search: stage 0 scores the first postings (position order) with no threshold, each later
    stage 32x more under the threshold the earlier stages produced (the k-th best score so far); stage 0 takes
    first * k postings.  No row may be
    reported twice across stages and the top-k of everything reported must be the oracle's top-k in the order
    (score desc, row asc), scores bit for bit."""
    n = ix["n"]
    full = _reference(ix, q_idx, w, 0, n, mask_bits, -np.inf)
    dfm = {int(t): int(d) for t, d in zip(ix["uniq"], ix["df"])}
    total = sum(dfm.get(t, 0) for t in q_idx)
    for k in ks:
        best = {}
        tau = np.float32(-np.inf)
        lo, hi = 0, first * k
        n_stage = 0
        while lo < total:
            got, _ = _run(emul, ix, q_idx, w, 0, n, mask_bits, tau, 512, 100, stage=(lo, hi))
            for r, s_ in got.items():
                assert r not in best, f"row {r} scored in two stages"
                assert s_ >= tau
                best[r] = s_
            ranked = sorted(best.values(), reverse=True)
            if len(ranked) >= k:
                tau = np.float32(max(tau, ranked[k - 1]))
            lo, hi = hi, hi * 32
            n_stage += 1
        assert n_stage >= 2
        want = sorted(((s_, -r) for r, s_ in full.items()), reverse=True)[:k]
        have = sorted(((s_, -r) for r, s_ in best.items()), reverse=True)[:k]
        assert [(float(a), -b) for a, b in have] == [(float(a), -b) for a, b in want], f"top {k}: (score, row)"
        assert all(best[-b].tobytes() == full[-b].tobytes() for _, b in want)


@pytest.mark.parametrize("seed", range(5))
def test_stages_score_every_row_once_and_reach_the_exact_top_k(emul, index, seed):
    ix = index
    q_idx, w = _query(ix, 700 + seed, (3, 12) if seed % 2 else (12, 40))
    rng = np.random.RandomState(seed)
    mask_bits = rng.randint(0, 2 ** 32, size=(ix["n"] + 31) // 32, dtype=np.uint64).astype(np.uint32) if seed % 2 else None
    _check_stages(emul, ix, q_idx, w, mask_bits, (5, 30))


@pytest.mark.parametrize("extra", [None, 3007])
@pytest.mark.parametrize("masked", [False, True])
def test_stages_keep_the_ties_at_the_cut_off(emul, ties_index, extra, masked):
    """On the tie-heavy corpus a later stage meets rows that EQUAL the threshold but have a lower id than the current
    k-th row: they belong in the top k.  Cut-offs inside tie groups (5, 30, 300) and among the score-0 rows."""
    ix = ties_index
    q_idx, w = _tie_query(ix, extra)
    rng = np.random.RandomState(4)
    mask_bits = rng.randint(0, 2 ** 32, size=(ix["n"] + 31) // 32, dtype=np.uint64).astype(np.uint32) if masked else None
    _check_stages(emul, ix, q_idx, w, mask_bits, (5, 30, 300))
    full = _reference(ix, q_idx, w, 0, ix["n"], mask_bits, -np.inf)
    k0 = sum(1 for s_ in full.values() if s_ > 0) + 3
    assert k0 < len(full)
    _check_stages(emul, ix, q_idx, w, mask_bits, (k0,), first=1)


@pytest.mark.parametrize("seed", range(5))
@pytest.mark.parametrize("masked", [False, True])
def test_k3h_hash_accumulate_matches_oracle(emul, index, seed, masked):
    """K3H (long queries): essential postings summed per row over row ranges, NE terms looked up best-first.  Candidates
    and score bits equal the oracle's for every threshold, segment and table capacity (a tiny capacity forces the
    range-halving path)."""
    ix = index
    n = ix["n"]
    q_idx, w = _query(ix, 900 + seed, (17, 64))
    rng = np.random.RandomState(seed)
    mask_bits = rng.randint(0, 2 ** 32, size=(n + 31) // 32, dtype=np.uint64).astype(np.uint32) if masked else None
    full = _reference(ix, q_idx, w, 0, n, mask_bits, -np.inf)
    ranked = sorted(full.values(), reverse=True)
    taus = [-np.inf, 0.0, float(ranked[min(len(ranked) - 1, 60)]), float(ranked[min(len(ranked) - 1, 5)]), float(ranked[0])]
    halved = 0
    for tau in taus:
        for (r0, r1) in ((0, n), (2048, n), (2048, 6144)):
            want = {r: s_ for r, s_ in full.items() if r0 <= r < r1 and s_ > np.float32(tau)}
            for max_post, budget, tabs, heavy in ((3072, 100, True, True), (40, 100, True, True), (3072, 20, False, False)):
                got, stats = _run(emul, ix, q_idx, w, r0, r1, mask_bits, np.float32(tau), 512, budget, tabs, heavy, mh_max_post=max_post)
                halved += int(stats[3])
                assert got.keys() == want.keys(), (tau, r0, r1, max_post, sorted(set(got) ^ set(want))[:10])
                bad = [r for r in want if got[r].tobytes() != want[r].tobytes()]
                assert not bad, f"score bits differ for rows {bad[:5]}"
    assert halved > 0
