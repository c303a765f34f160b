"""Exact score ties on every scoring path.  The engine and both oracles order a list by (score desc, row asc); these
tests hold every path to that order on a corpus where most scores tie:

* sparse: term A on the odd rows, term B on the even rows (equal df, so a query [A, B] weighs them alike), values
  from {0.5, 0.75, 1.0, 1.25}, every 37th row with a query-term value of 0.0 (score 0, still a candidate), extra terms
  with quantized values;
* dense: groups of duplicate rows (exact copies and copies scaled by powers of two, which give the same cosine bit for
  bit) across rows 127|128 (GEMM tile), 2047|2048 (first segment), 65535|65536 and the shard boundary of the two-shard
  case, and elsewhere.

Checks: the sparse list equals the C oracle's (rows, order and score bits), the fusion equals the Python oracle's fed
the GPU's own branch lists, and the dense list — scored in bf16, so against the GPU's own scores — is strictly ordered
by (score desc, row asc), gives every member of a duplicate group the same score, and returns a duplicate only after
every passing duplicate of a lower row id."""
import math

import numpy as np
import pytest

import _coded
import _data
from _parity import assert_same_list
from oracle import oracle as O
from oracle import oracle_c

pytestmark = pytest.mark.gpu

N, DIM = 70000, 64
TA, TB = 1000, 2000
EXTRA0, N_EXTRA = 3000, 200
SHARD = 40960                                  # row_base of the second shard in the two-shard case
FZ = {"weighted": 1, "rrf": 2}
N_SCOPES = 16


def _dup_groups(rng):
    """Row groups sharing one dense direction: 4 rows straddling each boundary, plus scattered groups."""
    groups = [list(range(b - 2, b + 2)) for b in (128, 2048, 65536, SHARD)]
    free = np.setdiff1d(np.arange(N), np.concatenate(groups))
    for _ in range(40):
        groups.append(sorted(rng.choice(free, size=int(rng.randint(2, 6)), replace=False).tolist()))
        free = np.setdiff1d(free, groups[-1])
    return groups


def make_tie_corpus(seed=29):
    rng = np.random.RandomState(seed)
    cents = rng.randn(32, DIM).astype(np.float32)
    dense = cents[rng.randint(0, 32, size=N)] + 0.7 * rng.randn(N, DIM).astype(np.float32)
    dense = _data.bf16_round(dense)
    groups = _dup_groups(rng)
    scale = np.float32([1.0, 2.0, 0.5, 1.0, 4.0, 0.25])
    for g in groups:
        for j, r in enumerate(g):
            dense[r] = dense[g[0]] * scale[j % len(scale)]          # powers of two: exact in bf16
    val = rng.choice(np.float32([0.5, 0.75, 1.0, 1.25]), size=N)
    val[::37] = 0.0
    rows = []
    for r in range(N):
        ex = EXTRA0 + rng.choice(N_EXTRA, size=int(rng.randint(1, 4)), replace=False)
        t = [TA if r % 2 else TB] + ex.tolist()
        v = [float(val[r])] + rng.choice([0.5, 1.0, 1.5], size=len(ex)).tolist()
        rows.append((t, v))
    for g in groups:        # duplicates share the sparse vector of their group's first row of the same parity (df stays equal)
        for r in g:
            rows[r] = rows[next(x for x in g if x % 2 == r % 2)]
    order = [np.argsort(t) for t, _ in rows]
    indptr = np.zeros(N + 1, np.int64)
    indptr[1:] = np.cumsum([len(t) for t, _ in rows])
    terms = np.concatenate([np.asarray(t, np.uint32)[o] for (t, _), o in zip(rows, order)])
    vals = np.concatenate([np.asarray(v, np.float32)[o] for (_, v), o in zip(rows, order)])
    scope = rng.randint(0, N_SCOPES, size=N).astype(np.uint32)
    created = np.full(N, _coded.TS_MISSING, np.int64)
    modified = rng.randint(1500000000, 1700000000, size=N).astype(np.int64)
    group_of = {r: gi for gi, g in enumerate(groups) for r in g}
    return dict(dense=dense, csr=(indptr, terms, vals), scope=scope, created=created, modified=modified,
                groups=groups, group_of=group_of, rng_seed=seed)


def make_queries(c, B, seed):
    """B queries cycling through the tie patterns; the dense part aims at a duplicate group."""
    rng = np.random.RandomState(seed)
    kinds = [
        ([TA, TB], [1.0, 1.0]),
        ([TA, TB, EXTRA0 + 7], [1.0, 1.0, 1.0]),
        ([TA], [1.0]),
        ([EXTRA0 + 3, EXTRA0 + 11], [1.0, 1.0]),
        ([TA, TB, EXTRA0 + 5], [1.0, 1.0, -0.5]),            # a negative weight: K3's exact path
        ([TB, TA, EXTRA0 + 9, EXTRA0 + 13], [1.0, 1.0, 0.5, 0.5]),
    ]
    Q, SP = [], []
    for i in range(B):
        g = c["groups"][i % len(c["groups"])]
        v = c["dense"][g[0]] / np.linalg.norm(c["dense"][g[0]])
        q = v + 0.3 * rng.randn(DIM).astype(np.float32) / np.sqrt(DIM)
        Q.append(_data.bf16_round((q / np.linalg.norm(q)).astype(np.float32)))
        SP.append(kinds[i % len(kinds)])
    return np.stack(Q), SP


@pytest.fixture(scope="module")
def tw():
    from voitta_rag_b200 import engine
    c = make_tie_corpus()
    ix = engine.Index(DIM)
    ix.upsert(c["dense"], c["csr"], c["scope"], c["created"], c["modified"])
    cc = oracle_c.CorpusC(c["dense"], c["csr"], c["scope"], c["created"], c["modified"])
    yield dict(c, ix=ix, cc=cc, engine=engine)
    ix.close()


def _fusion_bit_exact(got, i, limit, fusion, w):
    d = [O.ScoredPoint(str(r), s, {}, r) for r, s in got.branch(i, "dense")]
    s = [O.ScoredPoint(str(r), sc, {}, r) for r, sc in got.branch(i, "sparse")]
    want = O.reciprocal_rank_fusion([d, s], limit) if fusion == "rrf" else O.weighted_fusion(d, s, limit, w)
    assert [(int(pid), sc) for pid, sc, _ in want] == got.hits(i), f"fusion {fusion} q{i}"


def _dense_ties_hold(gd, c, passing, what):
    keys = [(-s, r) for r, s in gd]
    assert keys == sorted(keys) and len(set(r for r, _ in gd)) == len(gd), f"{what}: not strictly (score desc, row asc): {gd[:12]}"
    pos = {r: j for j, (r, _) in enumerate(gd)}
    for r, s in gd:
        gi = c["group_of"].get(r)
        if gi is None:
            continue
        for r2 in c["groups"][gi]:
            if r2 in pos:
                assert np.float32(gd[pos[r2]][1]).tobytes() == np.float32(s).tobytes(), \
                    f"{what}: duplicates {r2} and {r} scored {gd[pos[r2]][1]!r} and {s!r}"
            elif r2 < r:
                assert not passing[r2], f"{what}: duplicate {r} returned without the lower duplicate {r2}"


def run_and_check(w, Q, SP, filters=None, filter_of=None, limit=10, kprime=30, fusion="rrf", sparse_weight=0.3,
                  cc=None, ix=None, alive=None, what=""):
    eng = w["engine"]
    ix = ix or w["ix"]
    cc = cc or w["cc"]
    gf = None if filters is None else [eng.Filter(*f) for f in filters]
    got = ix.search_batch(Q, SP, gf, filter_of, limit=limit, kprime=kprime, fusion=fusion,
                          sparse_weight=sparse_weight, branches=True)
    want = cc.search_batch(Q, SP, filters, filter_of, limit=limit, kprime=kprime, fusion=FZ[fusion],
                           sparse_weight=sparse_weight)
    coded = dict(scope=w["scope"], created=w["created"], modified=w["modified"])
    for i in range(len(Q)):
        ws = [(int(want["sparse_rows"][i, j]), float(want["sparse_scores"][i, j])) for j in range(want["sparse_counts"][i])]
        assert_same_list(got.branch(i, "sparse"), ws, what=f"{what} sparse q{i}")
        _fusion_bit_exact(got, i, limit, fusion, sparse_weight)
        f = None if filters is None else (filters[filter_of[i]] if filter_of[i] >= 0 else None)
        passing = _coded.passing_rows(coded, f, alive)
        _dense_ties_hold(got.branch(i, "dense"), w, passing, f"{what} dense q{i}")
    return got


OPTION_SETS = {
    "default": {},
    "ms_staged0": {"ms_staged": 0},
    "sparse_ms0": {"sparse_ms": 0},
    "sparse_mh1": {"sparse_mh": 1, "ms_max_terms": 2},        # queries of 3+ terms go to K3H
    "safe_mode": {"safe_mode": 1},
}
DEFAULTS = {"ms_staged": 1, "sparse_ms": 1, "sparse_mh": 0, "ms_max_terms": 256, "safe_mode": 0}


@pytest.mark.parametrize("B", [1, 8, 320])
@pytest.mark.parametrize("opts", list(OPTION_SETS))
def test_ties_on_every_path(tw, B, opts):
    """B = 1: K1F; B = 8: resident K2 (bf16x2); B = 320: K2T — with K3M staged (default), per segment, off (K3), K3H
    for the longer queries, and the safe mode.  Both fusions."""
    ix = tw["ix"]
    Q, SP = make_queries(tw, B, seed=B)
    try:
        for k, v in OPTION_SETS[opts].items():
            ix.set_option(k, v)
        for fusion in ("rrf", "weighted"):
            run_and_check(tw, Q, SP, fusion=fusion, what=f"B={B} {opts} {fusion}")
            if B == 1 and opts != "safe_mode":
                assert ix.stats()["last_dense_path"] == 3            # K1F
    finally:
        for k, v in DEFAULTS.items():
            ix.set_option(k, v)


@pytest.mark.parametrize("B", [8, 320])
def test_ties_with_row_selection(tw, B):
    """K2 / K2T over the compacted copy of the rows that pass a batch-wide filter (forced on, small segments too)."""
    ix = tw["ix"]
    Q, SP = make_queries(tw, B, seed=100 + B)
    bits = np.uint32([0b0101_0101_0101_0111])
    flt = [(bits, 2, 1550000000, 1700000000)]
    fo = np.zeros(B, np.int32)
    try:
        ix.set_option("dense_compact", 100)
        ix.set_option("dense_compact_min_rows", 1024)
        run_and_check(tw, Q, SP, flt, fo, what=f"row selection B={B}")
    finally:
        ix.set_option("dense_compact", -1)
        ix.set_option("dense_compact_min_rows", 1 << 18)


def test_ties_with_per_query_filters(tw):
    """Every query its own scope set: the tie groups are cut differently per query."""
    B = 40
    Q, SP = make_queries(tw, B, seed=7)
    rng = np.random.RandomState(8)
    flts = [(np.uint32([int(rng.randint(1, 1 << N_SCOPES))]), 0, _coded.TS_MIN, _coded.TS_MAX) for _ in range(B)]
    fo = np.arange(B, dtype=np.int32)
    fo[::5] = -1
    for fusion in ("rrf", "weighted"):
        run_and_check(tw, Q, SP, flts, fo, fusion=fusion, what=f"per-query filters {fusion}")


def test_ties_with_delta_rows_and_deletes(tw):
    """Rows appended after the index build (scored by K3D) tie with indexed rows; deletes inside tie groups and
    duplicate groups."""
    eng = tw["engine"]
    ip, tm, vl = tw["csr"]
    nb = N - 3000
    ix = eng.Index(DIM)
    try:
        ix.upsert(tw["dense"][:nb], (ip[:nb + 1], tm[:ip[nb]], vl[:ip[nb]]), tw["scope"][:nb], tw["created"][:nb], tw["modified"][:nb])
        Q, SP = make_queries(tw, 8, seed=11)
        ix.search_batch(Q, SP, limit=10)                               # builds the inverted index over [0, nb)
        ix.upsert(tw["dense"][nb:], (ip[nb:] - ip[nb], tm[ip[nb]:], vl[ip[nb]:]), tw["scope"][nb:], tw["created"][nb:], tw["modified"][nb:])
        assert ix.stats()["n_rows"] == N
        for B in (1, 8):
            Qb, SPb = make_queries(tw, B, seed=20 + B)
            run_and_check(tw, Qb, SPb, ix=ix, what=f"delta B={B}")
        # deletes: low rows of the top tie groups, and the lowest member of every duplicate group
        dead = np.array(sorted(set([1, 2, 3, 5, 8, 9, 11, 14] + [g[0] for g in tw["groups"]])), np.uint64)
        ix.delete_rows(dead)
        alive = np.ones(N, np.uint8)
        alive[dead.astype(np.int64)] = 0
        cc = oracle_c.CorpusC(tw["dense"], tw["csr"], tw["scope"], tw["created"], tw["modified"], alive)
        for B in (1, 8, 320):
            Qb, SPb = make_queries(tw, B, seed=30 + B)
            run_and_check(tw, Qb, SPb, ix=ix, cc=cc, alive=alive, what=f"deletes B={B}")
    finally:
        ix.close()


def test_tie_flood_overflows_and_stays_exact():
    """More rows tied at the cut-off than a list holds: every row scores the same on [A, B], so after stage 0 every
    later posting ties with the threshold and is appended.  A batch of 320 gets lists of 49152 slots (8 sub-ranges);
    the 70k tied rows overflow them, the library re-runs the batch in safe mode, and the answer is exact."""
    from voitta_rag_b200 import engine
    n = N
    rng = np.random.RandomState(3)
    dense = _data.bf16_round(rng.randn(n, DIM).astype(np.float32))
    indptr = np.arange(n + 1, dtype=np.int64)
    terms = np.where(np.arange(n) % 2 == 1, TA, TB).astype(np.uint32)
    vals = np.ones(n, np.float32)
    ix = engine.Index(DIM)
    try:
        ix.upsert(dense, (indptr, terms, vals))
        cc = oracle_c.CorpusC(dense, (indptr, terms, vals))
        B = 320
        Q = _data.bf16_round(rng.randn(B, DIM).astype(np.float32))
        SP = [([TA, TB], [1.0, 1.0])] * B
        before = ix.stats()["overflow_reruns"]
        got = ix.search_batch(Q, SP, limit=10, kprime=30, fusion="rrf", branches=True)
        assert ix.stats()["overflow_reruns"] == before + 1
        want = cc.search_batch(Q, SP, limit=10, kprime=30, fusion=2)
        for i in range(B):
            ws = [(int(want["sparse_rows"][i, j]), float(want["sparse_scores"][i, j])) for j in range(want["sparse_counts"][i])]
            assert [r for r, _ in ws] == list(range(30))
            assert_same_list(got.branch(i, "sparse"), ws, what=f"flood sparse q{i}")
            _fusion_bit_exact(got, i, 10, "rrf", 0.1)
    finally:
        ix.close()


def test_ties_across_two_shards(tw):
    """Rows 0..SHARD-1 and SHARD.. on two indexes: shard 0 holds many rows that tie with shard 1's k'-th best.  The
    merged answer equals the single index's and the oracle's, without and with the threshold exchange (which must
    import the next float below the best k'-th, or shard 0 drops its tied rows of lower global id)."""
    import torch
    eng = tw["engine"]
    ip, tm, vl = tw["csr"]
    h = SHARD
    a = eng.Index(DIM, row_base=0)
    b = eng.Index(DIM, row_base=h)
    try:
        a.upsert(tw["dense"][:h], (ip[:h + 1], tm[:ip[h]], vl[:ip[h]]), tw["scope"][:h], tw["created"][:h], tw["modified"][:h])
        b.upsert(tw["dense"][h:], (ip[h:] - ip[h], tm[ip[h]:], vl[ip[h]:]), tw["scope"][h:], tw["created"][h:], tw["modified"][h:])
        B, limit, k = 8, 10, 30
        Q, SP = make_queries(tw, B, seed=41)
        # global IDF applied here, so that the shards, the single index and the oracle all take the same fp64 weights
        SPW = []
        for idx, val in SP:
            t = np.asarray(idx, np.uint32)
            (dfa, na), (dfb, nb_) = a.term_stats(t), b.term_stats(t)
            NL = na + nb_
            SPW.append((idx, [float(v) * math.log((NL - float(d) + 0.5) / (float(d) + 0.5) + 1.0) for v, d in zip(val, dfa + dfb)]))
        fo = np.zeros(B, np.int32)
        flt = [(np.uint32([0xFFFF]), 0, _coded.TS_MIN, _coded.TS_MAX)]
        gf = [eng.Filter(*flt[0])]
        for fusion in ("rrf", "weighted"):
            single = tw["ix"].search_batch(Q, SPW, gf, fo, limit=limit, kprime=k, fusion=fusion, apply_idf=False, branches=True)
            want = tw["cc"].search_batch(Q, SPW, flt, fo, limit=limit, kprime=k, fusion=FZ[fusion], apply_idf=False)
            bufs = [torch.zeros(eng.Index.cand_block_words(B, k), dtype=torch.int64, device="cuda") for _ in range(2)]
            a.search_local(bufs[0].data_ptr(), Q, SPW, gf, fo, limit=limit, kprime=k, fusion=fusion)
            b.search_local(bufs[1].data_ptr(), Q, SPW, gf, fo, limit=limit, kprime=k, fusion=fusion)
            torch.cuda.synchronize()
            merged = a.merge_fuse(torch.cat(bufs).data_ptr(), 2, Q, SPW, limit=limit, kprime=k, fusion=fusion, branches=True)
            staged, taus = [], []
            for sh in (a, b):
                staged.append(sh.stage(Q, SPW, gf, fo, limit=limit, kprime=k, fusion=fusion, apply_idf=False, branches=True))
                sh.run_local_begin()
                t = torch.zeros(2 * B, dtype=torch.float32, device="cuda")
                sh.tau_export(t.data_ptr())
                taus.append(t)
            torch.cuda.synchronize()
            tmax = torch.maximum(taus[0], taus[1])
            torch.cuda.synchronize()
            for sh, buf in zip((a, b), bufs):
                sh.tau_import(tmax.data_ptr())
                sh.run_local(buf.data_ptr())
            torch.cuda.synchronize()
            a.run_fuse(2, torch.cat(bufs).data_ptr())
            exchanged = a.fetch(staged[0])
            for name, res in (("merged", merged), ("threshold exchange", exchanged)):
                for i in range(B):
                    ws = [(int(want["sparse_rows"][i, j]), float(want["sparse_scores"][i, j])) for j in range(want["sparse_counts"][i])]
                    assert_same_list(res.branch(i, "sparse"), ws, what=f"{name} {fusion} sparse q{i}")
                    assert res.branch(i, "sparse") == single.branch(i, "sparse")
                    _fusion_bit_exact(res, i, limit, fusion, 0.1)
                    _dense_ties_hold(res.branch(i, "dense"), tw, _coded.passing_rows(dict(scope=tw["scope"], created=tw["created"], modified=tw["modified"]), flt[0]), f"{name} dense q{i}")
                for nm in ("rows", "counts", "dense_rows", "dense_scores", "dense_counts"):
                    assert np.array_equal(getattr(res, nm), getattr(single, nm)), (name, fusion, nm)
    finally:
        a.close()
        b.close()
