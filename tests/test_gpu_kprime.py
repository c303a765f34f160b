"""Every search path held to the oracle across the whole k' range the API accepts, 1 .. VB_MAX_KPRIME = 1024.

The service asks for k' = 3 * limit on a hybrid search (limit up to 341) and k' = limit on a dense-only one (limit up
to 1024).  Several mechanisms change regime as k' grows: the compaction's small path (<= VB_SORT_MAX = 2048 live keys)
against its histogram selection and the refinement inside a crowded pivot bin, K1F at its per-CTA capacity
(k' = VB_K1F_CAP / 2), the list capacity and the K3M stage sizes derived from k', the 2k' candidates of K4, the G*k'
keys of a shard merge, and lists shorter than k'.  The checks are those of test_gpu_engine.py / test_gpu_ties.py:

* sparse lists bit-equal to the C oracle (rows, order, score bits, list length);
* K4 bit-equal to the Python oracle's fusion fed the GPU's own branch lists;
* dense lists by assert_same_ranking at the path's tolerance (K1 / K1F 1e-5, K2 with a bf16x2 query 2e-5), or, on
  K2T (plain bf16 query, 1e-3), by assert_topk_valid against the full score vector;
* stats(): the dense path (3 = K1F, 1 = K1, 2 = K2 / K2T), the number of dense passes, and whether the safe-mode
  re-run happened — a case that drifts onto another path fails.
"""
import math

import numpy as np
import pytest

import _coded
import _data
from _parity import assert_same_list, assert_same_ranking, assert_topk_valid
from oracle import oracle as O
from oracle import oracle_c

pytestmark = pytest.mark.gpu

N, DIM = 200_000, 64
N_DELTA = 6000                     # rows upserted after the inverted index is built: scored by K3D
FZ = {"weighted": 1, "rrf": 2, "dense": 0}
DEFAULTS = {"k1f": 1, "safe_mode": 0, "dense_path": 0, "sparse_dense": 1}
KPRIMES = [1, 2, 31, 32, 33, 300, 683, 1023, 1024]


def _csr_slice(csr, lo, hi):
    ip, tm, vl = csr
    return (ip[lo:hi + 1] - ip[lo], tm[ip[lo]:ip[hi]], vl[ip[lo]:ip[hi]])


def _lst(want, branch, i):
    pre = "" if branch == "fused" else branch + "_"
    return [(int(want[pre + "rows"][i, j]), float(want[pre + "scores"][i, j])) for j in range(want[pre + "counts"][i])]


def _fusion_bit_exact(got, i, limit, fusion, w, what):
    d = [O.ScoredPoint(str(r), s, {}, r) for r, s in got.branch(i, "dense")]
    s = [O.ScoredPoint(str(r), sc, {}, r) for r, sc in got.branch(i, "sparse")]
    want = O.reciprocal_rank_fusion([d, s], limit) if fusion == "rrf" else O.weighted_fusion(d, s, limit, w)
    assert [(int(pid), sc) for pid, sc, _ in want] == got.hits(i), f"{what}: K4 q{i}"


def _strictly_ordered(lst, what):
    keys = [(-s, r) for r, s in lst]
    assert keys == sorted(keys) and len({r for r, _ in lst}) == len(lst), f"{what}: not strictly (score desc, row asc)"


@pytest.fixture(scope="module")
def kw():
    """200k x 64 hybrid corpus: 194k rows indexed, 6k appended after the index build (K3D), 3000 rows deleted."""
    from voitta_rag_b200 import engine
    corpus = _data.make_corpus(seed=41, n=N, dim=DIM, n_index=6, per_index=6, vocab=3000)
    coded = _coded.code_corpus(corpus)
    queries = _data.make_queries(seed=43, corpus=corpus, nq=320)
    nb = N - N_DELTA
    ix = engine.Index(DIM)
    ix.upsert(coded["dense"][:nb], _csr_slice(coded["csr"], 0, nb), coded["scope"][:nb], coded["created"][:nb],
              coded["modified"][:nb])
    ix.search_batch(np.stack([q for q, _ in queries[:2]]), [s for _, s in queries[:2]], limit=10)   # builds the index
    ix.upsert(coded["dense"][nb:], _csr_slice(coded["csr"], nb, N), coded["scope"][nb:], coded["created"][nb:],
              coded["modified"][nb:])
    assert ix.stats()["delta_rows"] == N_DELTA and ix.stats()["index_builds"] == 1
    rng = np.random.RandomState(44)
    dead = rng.choice(N, size=3000, replace=False)
    ix.delete_rows(dead)
    alive = np.ones(N, np.uint8)
    alive[dead] = 0
    cc = oracle_c.CorpusC(coded["dense"], coded["csr"], coded["scope"], coded["created"], coded["modified"], alive)
    # a query longer than 16 terms (K3M's long-query budget) and one with a negative weight (K3's exact path)
    r_long = next(r for r in range(N) if len(corpus["sparse"][r][0]) >= 20)
    t_long = list(corpus["sparse"][r_long][0]) + [int(corpus["term_ids"][7])]
    t_long = list(dict.fromkeys(t_long))
    assert len(t_long) > 16
    q_neg, (t_neg, _) = queries[1]
    special = [(queries[0][0], (t_long, [1.0] * len(t_long))), (q_neg, (t_neg, [-0.5] + [1.0] * (len(t_neg) - 1)))]
    # filters: about half the rows (a modified-date cut at the median), a few hundred rows (< k' for k' >= 683), and
    # scope sets for the per-query batch
    mod = coded["modified"]
    present = np.sort(mod[(mod != _coded.TS_MISSING) & (alive == 1)])
    half = (None, 2, int(present[len(present) // 2]), _coded.TS_MAX)
    few = (None, 2, int(present[40000]), int(present[40300]))
    sl = coded["scope_list"]
    folders = [f for f, _ in sl]
    incl = (_coded.scope_bits(sl, include=folders[:5]), 0, _coded.TS_MIN, _coded.TS_MAX)
    excl = (_coded.scope_bits(sl, exclude=folders[:2], disabled=["root3"]), 1, 1450000000, _coded.TS_MAX)
    n_pass = {name: int(_coded.passing_rows(coded, f, alive).sum()) for name, f in (("half", half), ("few", few))}
    assert 0.35 * N < n_pass["half"] < 0.55 * N, n_pass
    assert 100 < n_pass["few"] < 683, n_pass
    v = coded["dense"].astype(np.float64)
    xn = v / np.linalg.norm(v, axis=1, keepdims=True)
    yield dict(engine=engine, ix=ix, cc=cc, coded=coded, corpus=corpus, alive=alive, queries=queries, special=special,
               flt={"half": half, "few": few, "incl": incl, "excl": excl}, xn=xn)
    ix.close()


def _filters(w, kind, B):
    if kind == "none":
        return None, None
    if kind == "perq":
        fl = [w["flt"][k] for k in ("half", "few", "incl", "excl")]
        return fl, (np.arange(B) % (len(fl) + 1) - 1).astype(np.int32)          # -1 = unfiltered
    return [w["flt"][kind]], np.zeros(B, np.int32)


def _check(w, got, want, Q, kprime, limit, fusion, tol, fl, fo, what, sparse_weight=0.1):
    """tol None: plain bf16 query (K2T) — properties for every list, the full score vector for every 16th."""
    for i in range(len(Q)):
        gd, wd = got.branch(i, "dense"), _lst(want, "dense", i)
        f = None if fl is None or fo[i] < 0 else fl[fo[i]]
        passing = _coded.passing_rows(w["coded"], f, w["alive"])
        if tol is not None:
            assert_same_ranking(gd, wd, rel_tol=tol, abs_tol=tol, what=f"{what} dense q{i}")
        else:
            assert len(gd) == len(wd), f"{what} dense q{i}: length {len(gd)} != {len(wd)}"
            _strictly_ordered(gd, f"{what} dense q{i}")
            assert all(passing[r] for r, _ in gd), f"{what} dense q{i}: a row fails the filter or is deleted"
            if i % 16 == 0:
                q = np.asarray(Q[i], np.float64)
                scores = w["xn"] @ (q / np.linalg.norm(q))
                assert_topk_valid(gd, scores, passing.astype(bool), kprime, rel_tol=1e-3, abs_tol=1e-3, what=f"{what} dense q{i}")
        if fusion == "dense":
            assert got.hits(i) == gd[:limit], f"{what}: dense-only hits q{i}"
            continue
        assert_same_list(got.branch(i, "sparse"), _lst(want, "sparse", i), what=f"{what} sparse q{i}")
        _fusion_bit_exact(got, i, limit, fusion, sparse_weight, what)
        if tol is not None and [r for r, _ in gd] == [r for r, _ in wd]:
            # same dense input as the oracle's (up to fp32 summation error): the fused lists agree too
            assert_same_ranking(got.hits(i), _lst(want, "fused", i), rel_tol=10 * tol, abs_tol=10 * tol, what=f"{what} fused q{i}")


# (name, B, queries, options, dense path, tiled K2, filter, k' values) — a covering subset of k' x limit x B x path x
# filter, one row per regime:
SWEEP = [
    # B = 1, K1F (the default for single queries): every k' of the range, no filter and ~50 % alternating
    ("b1_k1f", 1, "plain", {}, 3, False, None, KPRIMES),
    # the K3M long-query budget and K3's exact path (negative weight) at the top of the range
    ("b1_long", 1, "long", {}, 3, False, "half", [1024]),
    ("b1_negative", 1, "negative", {}, 3, False, "none", [1024]),
    # B = 1, K1 in row segments (k1f = 0): seg_ratio 128, the first segment in direct slots; a filter that passes
    # fewer rows than k' (short lists, tau at -inf through every segment)
    ("b1_k1", 1, "plain", {"k1f": 0}, 1, False, "few", [33, 1024]),
    # B = 1 in safe mode: segments of cand_cap - k' rows, one sub-range per list
    ("b1_safe", 1, "plain", {"safe_mode": 1}, 1, False, "half", [1024]),
    # B = 3 (B <= 4: seg_ratio 128, lists of 16 * 128 * k' slots), resident K2 with a bf16x2 query
    ("b3_k2", 3, "plain", {}, 2, False, "none", [32, 683, 1024]),
    # B = 8, the largest K1F batch (dense_path = 1), per-query filters; k' = 1024 runs K1F at its buffer bound
    ("b8_k1f", 8, "plain", {"dense_path": 1}, 3, False, "perq", [1023, 1024]),
    # B = 9, one past K1F: K1 in row segments
    ("b9_k1", 9, "plain", {"dense_path": 1}, 1, False, "half", [1024]),
    # B = 40, resident K2 (bf16x2); the stage ratio sits at its floor of 32 at k' = 1024; long and negative queries
    # ride in the batch (K3 direct segment + K3M stages)
    ("b40_k2", 40, "mixed", {}, 2, False, "perq", [31, 300, 1024]),
    ("b40_safe", 40, "mixed", {"safe_mode": 1}, 2, False, "few", [1024]),
    # B = 320 > the resident sub-batch of 256 queries at d_pad 64: K2T (one pass) with a plain bf16 query
    ("b320_k2t", 320, "plain", {}, 2, True, "half", [1024]),
]


def _queries(w, kind, B):
    if kind == "long":
        return w["special"][:1]
    if kind == "negative":
        return w["special"][1:]
    if kind == "mixed":
        return w["special"] + w["queries"][2:B]
    return w["queries"][:B]


@pytest.mark.parametrize("name,B,qkind,opts,path,tiled,fkind,kps", SWEEP, ids=[s[0] for s in SWEEP])
def test_kprime_sweep_against_oracle(kw, name, B, qkind, opts, path, tiled, fkind, kps):
    ix, eng = kw["ix"], kw["engine"]
    qs = _queries(kw, qkind, B)
    Q = np.stack([q for q, _ in qs])
    SP = [s for _, s in qs]
    tol = None if tiled else (2e-5 if path == 2 else 1e-5)
    try:
        for k, v in opts.items():
            ix.set_option(k, v)
        for j, kp in enumerate(kps):
            fk = fkind or ("none", "half")[j % 2]
            fl, fo = _filters(kw, fk, B)
            gf = None if fl is None else [eng.Filter(*f) for f in fl]
            runs = [("dense", kp)]
            if kp // 3 >= 1:
                runs.append((("weighted", "rrf")[j % 2], kp // 3))
            runs.append((("rrf", "weighted")[j % 2], kp))
            for fusion, limit in runs:
                what = f"{name} k'={kp} limit={limit} {fusion} filter={fk}"
                before = ix.stats()["overflow_reruns"]
                sp = None if fusion == "dense" else SP
                got = ix.search_batch(Q, sp, gf, fo, limit=limit, kprime=kp, fusion=fusion, branches=True)
                st = ix.stats()
                assert st["last_dense_path"] == path, (what, st)
                if path == 2:
                    # one pass: K2T for B > 256 (the resident kernel would take two), one resident sub-batch below
                    assert st["last_dense_passes"] == 1 and (B > 256) == tiled, (what, st)
                assert st["overflow_reruns"] == before and st["last_overflow_lists"] == 0, (what, st)
                assert got.dense_rows.shape == (B, kp) and got.rows.shape == (B, limit)
                want = kw["cc"].search_batch(Q, sp, fl, fo, limit=limit, kprime=kp, fusion=FZ[fusion])
                _check(kw, got, want, Q, kp, limit, fusion, tol, fl, fo, what)
                if fk == "few":          # fewer passing rows than k': every one of them comes back
                    n_few = int(_coded.passing_rows(kw["coded"], kw["flt"]["few"], kw["alive"]).sum())
                    assert all(int(c) == min(kp, n_few) for c in got.dense_counts), what
    finally:
        for k in opts:
            ix.set_option(k, DEFAULTS[k])


# ---------------------------------------------------------------------------------------------------------------------
# Lists longer than the data
# ---------------------------------------------------------------------------------------------------------------------

def test_lists_longer_than_the_data():
    """333 rows (not a multiple of 32), 7 deleted, two exact duplicates, k' = 1024: every list stays short of k' through
    every segment and K3M stage (tau never leaves -inf).  Every live row comes back in (score desc, row asc) order, the
    sparse list equals the oracle's bit for bit, the fused list equals the oracle's."""
    from voitta_rag_b200 import engine
    rng = np.random.RandomState(333)
    n = 333
    dense = _data.bf16_round(rng.randn(n, DIM).astype(np.float32))
    vocab = np.arange(100, 120, dtype=np.uint32)
    rows = []
    for _ in range(n):
        t = np.sort(rng.choice(vocab, size=int(rng.randint(3, 7)), replace=False))
        rows.append((t, rng.choice(np.float32([0.5, 1.0, 1.5, 2.0]), size=len(t))))
    dense[200] = dense[10]
    rows[200] = rows[10]
    indptr = np.zeros(n + 1, np.int64)
    indptr[1:] = np.cumsum([len(t) for t, _ in rows])
    csr = (indptr, np.concatenate([t for t, _ in rows]).astype(np.uint32), np.concatenate([v for _, v in rows]).astype(np.float32))
    scope = rng.randint(0, 4, size=n).astype(np.uint32)
    ix = engine.Index(DIM)
    try:
        ix.upsert(dense, csr, scope)
        dead = np.array([0, 31, 32, 64, 150, 299, 332], np.uint64)
        ix.delete_rows(dead)
        alive = np.ones(n, np.uint8)
        alive[dead.astype(np.int64)] = 0
        cc = oracle_c.CorpusC(dense, csr, scope, None, None, alive)
        n_live = int(alive.sum())
        Q1 = _data.bf16_round(dense[10] + 0.2 * rng.randn(DIM).astype(np.float32))
        SP1 = ([100, 103, 111], [1.0, 1.0, 1.0])
        for B, opts, path, tol in ((1, {}, 3, 1e-5), (1, {"k1f": 0}, 1, 1e-5), (40, {}, 2, 2e-5)):
            Q = np.stack([Q1] + [_data.bf16_round(rng.randn(DIM).astype(np.float32)) for _ in range(B - 1)])
            SP = [SP1] + [(sorted(rng.choice(vocab, size=3, replace=False).tolist()), [1.0] * 3) for _ in range(B - 1)]
            try:
                for k, v in opts.items():
                    ix.set_option(k, v)
                for fusion, limit in (("dense", 1024), ("weighted", 341), ("rrf", 341)):
                    what = f"short lists B={B} {opts} {fusion}"
                    sp = None if fusion == "dense" else SP
                    got = ix.search_batch(Q, sp, limit=limit, kprime=1024, fusion=fusion, branches=True)
                    assert ix.stats()["last_dense_path"] == path and ix.stats()["last_overflow_lists"] == 0
                    want = cc.search_batch(Q, sp, limit=limit, kprime=1024, fusion=FZ[fusion])
                    for i in range(B):
                        gd = got.branch(i, "dense")
                        assert sorted(r for r, _ in gd) == np.flatnonzero(alive).tolist(), f"{what} q{i}: not every live row"
                        _strictly_ordered(gd, f"{what} dense q{i}")
                        pos = {r: s for r, s in gd}
                        assert np.float32(pos[10]).tobytes() == np.float32(pos[200]).tobytes(), what
                        assert_same_ranking(gd, _lst(want, "dense", i), rel_tol=tol, abs_tol=tol, what=f"{what} dense q{i}")
                        if fusion == "dense":
                            assert got.hits(i) == gd and len(gd) == n_live
                            continue
                        gs = got.branch(i, "sparse")
                        assert_same_list(gs, _lst(want, "sparse", i), what=f"{what} sparse q{i}")
                        assert len(gs) < 1024
                        _fusion_bit_exact(got, i, limit, fusion, 0.1, what)
                        assert_same_ranking(got.hits(i), _lst(want, "fused", i), rel_tol=10 * tol, abs_tol=10 * tol, what=f"{what} fused q{i}")
            finally:
                for k in opts:
                    ix.set_option(k, DEFAULTS[k])
    finally:
        ix.close()


# ---------------------------------------------------------------------------------------------------------------------
# The compaction's selection and refinement under a tie flood
# ---------------------------------------------------------------------------------------------------------------------

FLOOD_N = 60_000
FLOOD_BLOCKS = [(600, 3700), (20_000, 23_100)]      # 3100 + 3100 rows; the first straddles row 2048
TF, TG, TH = 5, 6, 7                                # the flood's term, a lower-scoring term, the 2200-row term
H_HIGH, H_TIE = 900, 1300


def _flood_corpus():
    rng = np.random.RandomState(2048)
    dense = _data.bf16_round(rng.randn(FLOOD_N, DIM).astype(np.float32))
    v = dense[FLOOD_BLOCKS[0][0]].copy()
    flood = np.concatenate([np.arange(a, b) for a, b in FLOOD_BLOCKS])
    dense[flood] = v
    rest = np.setdiff1d(np.arange(FLOOD_N), flood)
    g_rows = set(rng.choice(rest, size=3000, replace=False).tolist())
    h_rows = rng.choice(rest, size=H_HIGH + H_TIE, replace=False)
    h_val = {int(r): np.float32(2.0 + k / 1000.0) for k, r in enumerate(h_rows[:H_HIGH])}
    h_val.update({int(r): np.float32(1.0) for r in h_rows[H_HIGH:]})
    flood_set = set(flood.tolist())
    terms, vals, indptr = [], [], [0]
    for r in range(FLOOD_N):
        if r in flood_set:
            t, x = [TF, 1000], [1.0, 0.5]                 # bit-identical sparse vectors
        else:
            t = sorted(rng.choice(np.arange(1000, 1400), size=int(rng.randint(1, 4)), replace=False).tolist())
            x = rng.choice([0.5, 1.0, 1.5], size=len(t)).tolist()
            if r in h_val:
                t, x = [TH] + t, [float(h_val[r])] + x
            if r in g_rows:
                t, x = [TG] + t, [0.25] + x               # (TG < TH < 1000: indices stay ascending)
        terms += t
        vals += x
        indptr.append(len(terms))
    csr = (np.asarray(indptr, np.int64), np.asarray(terms, np.uint32), np.asarray(vals, np.float32))
    return dense, csr, v


def test_compaction_refines_a_tie_flood_down_to_the_row_bits():
    """6200 rows with bit-identical dense and sparse vectors (rows 600..3699 across the 2047|2048 boundary, and
    20000..23099), searched with the flood's own dense vector at k' in {1000, 1024}, B = 1 (K1F) and B = 40 (K2).

    Sparse, query [F, G]: K3M stage 0 scores the first 8192 postings in descending-bound order with no threshold —
    the 6200 postings of F (all the same score) and 1992 of G — so that stage's compaction holds 8192 live keys, four
    times VB_SORT_MAX: the general path, whose first digit puts every flood key in one pivot bin that must then be
    split by the row bits.  Sparse, query [H]: 2200 postings, 900 with distinct high values above 1300 tied at 1.0 —
    one compaction with 2200 live keys (just past VB_SORT_MAX, so the small path must give up) whose pivot bin holds
    the tie with 900 keys above it (2200 keys at or above the pivot: the bin must be refined).  Dense: the K1F merge
    holds one local top-k' per CTA, the resident K2 appends the 1652 flood rows past row 2048 to a list of k' keys
    whose threshold they tie — both far past 2048 keys of one score.

    The lowest row ids of the flood must fill the list exactly: nothing dropped, nothing duplicated."""
    from voitta_rag_b200 import engine
    dense, csr, v = _flood_corpus()
    ix = engine.Index(DIM)
    try:
        ix.upsert(dense, csr)
        cc = oracle_c.CorpusC(dense, csr)
        lo = FLOOD_BLOCKS[0][0]
        for B, path, tol in ((1, 3, 1e-5), (40, 2, 2e-5)):
            for sq in (([TF, TG], [1.0, 1.0]), ([TH], [1.0])):
                Q = np.stack([v] * B)
                SP = [sq] * B
                for kp in (1000, 1024):
                    what = f"flood B={B} terms={sq[0]} k'={kp}"
                    got = ix.search_batch(Q, SP, limit=kp // 3, kprime=kp, fusion="rrf", branches=True)
                    st = ix.stats()
                    assert st["last_dense_path"] == path and st["last_overflow_lists"] == 0, (what, st)
                    want = cc.search_batch(Q, SP, limit=kp // 3, kprime=kp, fusion=2)
                    for i in range(B):
                        gd = got.branch(i, "dense")
                        assert [r for r, _ in gd] == list(range(lo, lo + kp)), f"{what} dense q{i}: {gd[:3]} .. {gd[-3:]}"
                        assert len({np.float32(s).tobytes() for _, s in gd}) == 1, f"{what}: flood rows scored differently"
                        assert_same_ranking(gd, _lst(want, "dense", i), rel_tol=tol, abs_tol=tol, what=f"{what} dense q{i}")
                        ws = _lst(want, "sparse", i)
                        if sq[0][0] == TF:
                            assert [r for r, _ in ws] == list(range(lo, lo + kp))
                        assert_same_list(got.branch(i, "sparse"), ws, what=f"{what} sparse q{i}")
                        _fusion_bit_exact(got, i, kp // 3, "rrf", 0.1, what)
    finally:
        ix.close()


# ---------------------------------------------------------------------------------------------------------------------
# Overflow and the safe-mode re-run at k' = 1024
# ---------------------------------------------------------------------------------------------------------------------

def test_dense_overflow_at_kprime_1024_falls_back_to_safe_mode():
    """Scores strictly rising with the row id (the construction of test_overflow_falls_back_to_safe_mode_and_stays_exact),
    2.6M rows, k' = 1024 — every row of a segment beats the threshold, so a segment appends all its rows:

    * B = 1, K1 (k1f = 0): lists of 16 * 128 * k' = 2,097,152 slots, segments at 2048 * 128^i: the segment
      [262144, 2.6M) appends 2,337,856 keys > 2,097,152 slots;
    * B = 40, resident K2: lists of 417,792 slots (256 MB over 80 lists), segments at 2048 * 8^i: [131072, 1048576)
      appends 917,504 keys.

    Both overflow for certain, re-run in safe mode (segments of cand_cap - k' rows: no overflow) and stay exact."""
    from voitta_rag_b200 import engine
    n = 2_600_000
    theta = np.linspace(1.5, 0.05, n)
    dense = np.zeros((n, DIM), np.float32)
    dense[:, :2] = _data.bf16_round(np.stack([np.cos(theta), np.sin(theta)], axis=1).astype(np.float32))
    v = dense[:, :2].astype(np.float64)
    scores = (v[:, 0] / np.linalg.norm(v, axis=1)).astype(np.float32)
    ix = engine.Index(DIM)
    try:
        ix.upsert(dense)
        del dense
        q = np.zeros(DIM, np.float32)
        q[0] = 1.0
        everyone = np.ones(n, bool)
        for B, opts, path, tol in ((1, {"k1f": 0}, 1, 1e-5), (40, {}, 2, 2e-5)):
            for k, val in opts.items():
                ix.set_option(k, val)
            before = ix.stats()["overflow_reruns"]
            r = ix.search_batch(np.stack([q] * B), limit=1024, fusion="dense")
            st = ix.stats()
            for k in opts:
                ix.set_option(k, DEFAULTS[k])
            assert st["overflow_reruns"] == before + 1 and st["last_overflow_lists"] == 0, st
            assert st["last_dense_path"] == path, st
            for i in sorted({0, B - 1}):
                assert_topk_valid(r.hits(i), scores, everyone, 1024, rel_tol=tol, abs_tol=tol, what=f"ascending corpus B={B} q{i}")
    finally:
        ix.close()


def test_k3m_stage_overflow_at_kprime_1024_falls_back_to_safe_mode():
    """A K3M stage that appends more than the lists hold.  1M rows, one term on every 9th row (111,112 postings: fewer
    than 1/8 of the rows, so it is walked as postings, not read from a dense column), its value rising with the row
    id, so the best rows come last in posting order.  B = 320, k' = 1024: lists of max(2 * 32 * k', min(16 * 128 * k',
    256 MB / (640 lists * 8 B))) = 65,536 slots, 8 sub-ranges of 8192.  Stage 0 scores postings [0, 8192) with no
    threshold; the stage ratio is max(32, 65536 / (16 k')) = 32, so stage 1 scores postings [8192, 111112): every one
    of those 102,920 beats stage 0's threshold and is appended — more than the 65,536 slots of the whole list.

    The dense branch alone (random rows) does not overflow; the hybrid batch does, re-runs in safe mode (K3M per row
    segment of cand_cap - k' rows) and returns the exact sparse lists: the 1024 last rows of the term, best first,
    their values as scores (no IDF)."""
    from voitta_rag_b200 import engine
    rng = np.random.RandomState(9)
    n, B, kp, T = 1_000_000, 320, 1024, 77
    dense = _data.bf16_round(rng.randn(n, DIM).astype(np.float32))
    rows_t = np.arange(0, n, 9)
    val = (1.0 + rows_t / n).astype(np.float32)
    assert len(np.unique(val)) == len(val) and len(rows_t) * 8 < n
    has = np.zeros(n, bool)
    has[rows_t] = True
    counts = has.astype(np.int64) + 1                      # every row also carries one filler term
    indptr = np.zeros(n + 1, np.int64)
    np.cumsum(counts, out=indptr[1:])
    terms = np.empty(indptr[-1], np.uint32)
    vals = np.empty(indptr[-1], np.float32)
    terms[indptr[rows_t]] = T
    vals[indptr[rows_t]] = val
    filler = indptr[1:] - 1
    terms[filler] = 1000 + rng.randint(0, 5000, size=n)
    vals[filler] = 1.0
    ix = engine.Index(DIM)
    try:
        ix.upsert(dense, (indptr, terms, vals))
        Q = _data.bf16_round(rng.randn(B, DIM).astype(np.float32))
        before = ix.stats()["overflow_reruns"]
        ix.search_batch(Q, None, limit=kp, fusion="dense")
        assert ix.stats()["overflow_reruns"] == before
        SP = [([T], [1.0])] * B
        got = ix.search_batch(Q, SP, limit=kp // 3, kprime=kp, fusion="rrf", branches=True, apply_idf=False)
        st = ix.stats()
        assert st["overflow_reruns"] == before + 1 and st["last_overflow_lists"] == 0, st
        assert st["last_dense_path"] == 2 and st["last_dense_passes"] == 1, st
        want = [(int(r), float(s)) for r, s in zip(rows_t[::-1][:kp], val[::-1][:kp])]
        sparse_scores = np.full(n, -np.inf)
        sparse_scores[rows_t] = val
        norms = np.linalg.norm(dense, axis=1)
        for i in range(B):
            assert_same_list(got.branch(i, "sparse"), want, what=f"K3M overflow sparse q{i}")
            _fusion_bit_exact(got, i, kp // 3, "rrf", 0.1, "K3M overflow")
        for i in (0, B // 2, B - 1):
            assert_topk_valid(got.branch(i, "sparse"), sparse_scores, np.ones(n, bool), kp, rel_tol=0.0, what=f"K3M overflow q{i}")
            cos = (dense @ (Q[i] / np.linalg.norm(Q[i]))) / norms
            assert_topk_valid(got.branch(i, "dense"), cos, np.ones(n, bool), kp,
                              rel_tol=1e-3, abs_tol=1e-3, what=f"K3M overflow dense q{i}")
    finally:
        ix.close()


# ---------------------------------------------------------------------------------------------------------------------
# Shard merge at k' = 1024
# ---------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("G", [2, 8])
def test_sharded_merge_at_kprime_1024_equals_single_index(kw, G):
    """G row shards (search_local on each, candidates concatenated as the all-gather would, merge_fuse): with 8 shards
    the merge compacts 8 * 1024 = 8192 keys per list.  Global IDF applied by the caller, so that the single index and
    the shards take the same weights: branches and fused list bit-equal to the single index."""
    import torch
    eng, coded, alive = kw["engine"], kw["coded"], kw["alive"]
    B, kp, limit = 8, 1024, 341
    qs = kw["queries"][:B]
    Q = np.stack([q for q, _ in qs])
    SP = [s for _, s in qs]
    bounds = np.linspace(0, N, G + 1).astype(np.int64)
    shards = []
    try:
        for lo, hi in zip(bounds[:-1], bounds[1:]):
            sh = eng.Index(DIM, row_base=int(lo))
            sh.upsert(coded["dense"][lo:hi], _csr_slice(coded["csr"], lo, hi), coded["scope"][lo:hi], coded["created"][lo:hi],
                      coded["modified"][lo:hi])
            dead = np.flatnonzero(alive[lo:hi] == 0) + lo
            if len(dead):
                sh.delete_rows(dead.astype(np.uint64))
            shards.append(sh)
        SPW = []
        for idx, val in SP:
            t = np.asarray(idx, np.uint32)
            stats = [sh.term_stats(t) for sh in shards]
            df = sum(s[0].astype(np.int64) for s in stats)
            NL = sum(s[1] for s in stats)
            SPW.append((idx, [float(x) * math.log((NL - float(d) + 0.5) / (float(d) + 0.5) + 1.0) for x, d in zip(val, df)]))
        fk = "none" if G == 2 else "half"
        fl, fo = _filters(kw, fk, B)
        gf = None if fl is None else [eng.Filter(*f) for f in fl]
        words = eng.Index.cand_block_words(B, kp)
        for fusion in ("weighted", "rrf"):
            single = kw["ix"].search_batch(Q, SPW, gf, fo, limit=limit, kprime=kp, fusion=fusion, apply_idf=False, branches=True)
            gathered = torch.zeros(G * words, dtype=torch.int64, device="cuda")
            for r, sh in enumerate(shards):
                sh.search_local(gathered[r * words:].data_ptr(), Q, SPW, gf, fo, limit=limit, kprime=kp, fusion=fusion)
                assert sh.stats()["last_dense_path"] == 2
            torch.cuda.synchronize()
            merged = shards[0].merge_fuse(gathered.data_ptr(), G, Q, SPW, limit=limit, kprime=kp, fusion=fusion, branches=True)
            assert shards[0].stats()["last_overflow_lists"] == 0
            for name in ("rows", "scores", "counts", "dense_rows", "dense_scores", "dense_counts", "sparse_rows",
                         "sparse_scores", "sparse_counts"):
                assert np.array_equal(getattr(merged, name), getattr(single, name)), (G, fusion, name)
            assert all(int(c) == kp for c in merged.dense_counts)
            want = kw["cc"].search_batch(Q, SPW, fl, fo, limit=limit, kprime=kp, fusion=FZ[fusion], apply_idf=False)
            for i in range(B):
                assert_same_list(merged.branch(i, "sparse"), _lst(want, "sparse", i), what=f"G={G} {fusion} sparse q{i}")
                _fusion_bit_exact(merged, i, limit, fusion, 0.1, f"G={G}")
    finally:
        for sh in shards:
            sh.close()


# ---------------------------------------------------------------------------------------------------------------------
# The service boundary
# ---------------------------------------------------------------------------------------------------------------------

def test_vector_store_at_the_edges_of_the_kprime_range(monkeypatch):
    """VectorStoreService.search against oracle.OracleVectorStore on the same chunks: hybrid at limit 1 (k' = 3) and
    341 (k' = 1023), dense-only at limit 1024 — ids, order and scores.  A hybrid limit of 342 would need k' = 1026:
    refused with the library's message naming the cap, never answered with a shorter list."""
    from voitta_rag_b200 import engine
    from voitta_rag_b200 import vector_store as VS
    name = "gpu_kprime_edges"
    n, dim = 12_000, 64
    monkeypatch.setenv("QDRANT_COLLECTION", name)
    monkeypatch.setenv("EMBEDDING_DIMENSION", str(dim))
    VS._drop_collection(name)
    try:
        store = VS.VectorStoreService()
        corpus = _data.make_corpus(seed=17, n=n, dim=dim, n_index=6, per_index=6, vocab=2000)
        chunks = [(corpus["texts"][r], corpus["dense"][r].astype(float).tolist(), VS.ChunkMetadata(**corpus["metas"][r]))
                  for r in range(n)]
        sparse = [corpus["sparse"][r] for r in range(n)]
        ids = store.store_chunks(chunks, sparse)
        ref = O.OracleVectorStore(dim, fusion=store.fusion)
        ref.store_chunks(chunks, sparse, ids=ids)
        folders = sorted({m["folder_path"] for m in corpus["metas"]})
        qs = _data.make_queries(seed=6, corpus=corpus, nq=4)
        for qi, (q, sq) in enumerate(qs):
            ql = q.astype(float).tolist()
            kw = {} if qi % 2 == 0 else {"include_folders": folders[:12]}
            for limit, sp in ((1, sq), (341, sq), (1024, None)):
                what = f"service q{qi} limit={limit} {'hybrid' if sp else 'dense'} {kw}"
                got = store.search(ql, limit=limit, sparse_query=sp, **kw)
                assert store.client.stats()["last_dense_path"] == 3, what          # one query: K1F
                want = ref.search(ql, limit=limit, sparse_query=sp, **kw)
                assert len(got) == len(want) and (kw or len(got) == limit), what
                assert_same_ranking([(c.id, c.score) for c in got], [(c.id, c.score) for c in want], rel_tol=1e-5, abs_tol=1e-5, what=what)
                by_id = {c.id: c for c in want}
                for c in got:
                    if c.id in by_id:
                        assert c.text == by_id[c.id].text and vars(c.metadata) == vars(by_id[c.id].metadata), what
        q, sq = qs[0]
        with pytest.raises(engine.B200Error, match=r"kprime 1026 exceeds VB_MAX_KPRIME \(1024\)"):
            store.search(q.astype(float).tolist(), limit=342, sparse_query=sq)
        with pytest.raises(engine.B200Error, match=r"kprime 1025 exceeds VB_MAX_KPRIME \(1024\)"):
            store.search(q.astype(float).tolist(), limit=1025)
        ix = store.client
        with pytest.raises(engine.B200Error, match=r"kprime 1025 exceeds VB_MAX_KPRIME \(1024\)"):
            ix.search_batch(q[None, :], [sq], limit=10, kprime=1025)
        with pytest.raises(engine.B200Error, match=r"kprime \(9\) < limit \(10\)"):
            ix.search_batch(q[None, :], [sq], limit=10, kprime=9)
        assert engine.MAX_KPRIME == 1024
    finally:
        VS._drop_collection(name)
