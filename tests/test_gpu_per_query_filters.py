"""Per-query filters on the tensor-core paths: batches of up to 1024 distinct filters through K2T (query-tiled) and the
resident K2 over several sub-batches, the merging of unused and content-equal filters, the staged two-shard flow and
the drop-in VectorStoreService.search_batch(filters=...).  Each tile of queries carries its own filter table, so the
number of filters a batch holds is not bounded by the epilogue's per-tile cache of 256 mask words."""
import numpy as np
import pytest

import _data
from _parity import assert_same_ranking
from oracle import oracle as O
from oracle import oracle_c

pytestmark = pytest.mark.gpu

T0, T1 = 1420070400, 1767225600


def fusion_bit_exact(got, i, limit):
    d = [O.ScoredPoint(str(r), s, {}, r) for r, s in got.branch(i, "dense")]
    s = [O.ScoredPoint(str(r), sc, {}, r) for r, sc in got.branch(i, "sparse")]
    assert [(int(pid), sc) for pid, sc, _ in O.reciprocal_rank_fusion([d, s], limit)] == got.hits(i)


@pytest.fixture(scope="module")
def big():
    """150k x 768 hybrid corpus, 64 scopes, modified timestamps, 2 % of the rows deleted (so that unfiltered queries
    carry the alive-only filter)."""
    from voitta_rag_b200 import engine
    rng = np.random.RandomState(768)
    n, dim, B = 150_000, 768, 1024
    cents = rng.randn(256, dim).astype(np.float32)
    dense = _data.bf16_round(cents[rng.randint(0, 256, size=n)] + 0.7 * rng.randn(n, dim).astype(np.float32))
    vocab = np.unique(rng.randint(1, 2**31 - 1, size=8000).astype(np.int64))[:4000]
    p = 1.0 / np.arange(1, len(vocab) + 1) ** 1.07; p /= p.sum()
    picks = np.sort(rng.choice(len(vocab), size=(n, 10), p=p), axis=1)
    rows_terms = [np.unique(vocab[picks[r]]) for r in range(n)]
    indptr = np.zeros(n + 1, np.int64); np.cumsum([len(t) for t in rows_terms], out=indptr[1:])
    terms = np.concatenate(rows_terms).astype(np.uint32)
    vals = (0.5 + 1.5 * rng.rand(len(terms))).astype(np.float32)
    scope = rng.randint(0, 64, size=n).astype(np.uint32)
    modified = rng.randint(T0, T1, size=n).astype(np.int64)
    ix = engine.Index(dim)
    ix.upsert(dense, (indptr, terms, vals), scope, None, modified)
    dead = rng.choice(n, size=n // 50, replace=False)
    ix.delete_rows(dead)
    alive = np.ones(n, bool); alive[dead] = False
    cc = oracle_c.CorpusC(dense, (indptr, terms, vals), scope, None, modified, alive=alive.astype(np.uint8))
    qrows = rng.randint(0, n, size=B)
    Q = _data.bf16_round(dense[qrows] + 0.4 * rng.randn(B, dim).astype(np.float32))
    SP = [list(dict.fromkeys(rows_terms[r][:5].tolist() + [int(vocab[rng.randint(0, len(vocab))])])) for r in qrows]
    SP = [(t, [1.0] * len(t)) for t in SP]
    yield dict(engine=engine, ix=ix, cc=cc, dense=dense, scope=scope, modified=modified, alive=alive, Q=Q, SP=SP, B=B,
               indptr=indptr, terms=terms, vals=vals, n=n, dim=dim)
    ix.close()


def distinct_filters(count, seed):
    """`count` filters of distinct content: a random scope set and a date range each, selectivities from ~1 % to ~60 %."""
    rng = np.random.RandomState(seed)
    out = []
    for k in range(count):
        sel = float(np.exp(rng.uniform(np.log(0.01), np.log(0.6))))
        frac = rng.uniform(0.6, 1.0)
        m = int(np.clip(round(64 * sel / frac), 1, 64))
        bits = np.zeros(2, np.uint32)
        for s in rng.choice(64, size=m, replace=False):
            bits[s >> 5] |= np.uint32(1 << (s & 31))
        lo = T0 + int(rng.uniform(0, 1 - frac) * (T1 - T0)) + k          # + k: no two ranges are equal
        out.append((bits, 2, lo, lo + int(frac * (T1 - T0))))
    return out


def passes(w, f, rows):
    rows = np.asarray(rows, np.int64)
    ok = w["alive"][rows]
    if f is not None:
        sc = w["scope"][rows]
        ok &= ((f[0][sc >> 5] >> (sc & 31)) & 1).astype(bool) & (w["modified"][rows] >= f[2]) & (w["modified"][rows] <= f[3])
    return ok


def check_batch(w, got, fl, fo, what, limit=100):
    """Oracle on a 96-query subset; every query: unique rows in score order, each passing its own filter and alive."""
    B = w["B"]
    sub = np.sort(np.random.RandomState(5).choice(B, size=96, replace=False))
    want = w["cc"].search_batch(w["Q"][sub], [w["SP"][i] for i in sub], fl, fo[sub], limit=limit, kprime=3 * limit, fusion=2)
    for j, i in enumerate(sub):
        wd = [(int(want["dense_rows"][j, t]), float(want["dense_scores"][j, t])) for t in range(want["dense_counts"][j])]
        assert_same_ranking(got.branch(i, "dense"), wd, rel_tol=1e-3, abs_tol=1e-3, what=f"{what} dense q{i}")
        ws = [(int(want["sparse_rows"][j, t]), float(want["sparse_scores"][j, t])) for t in range(want["sparse_counts"][j])]
        assert_same_ranking(got.branch(i, "sparse"), ws, rel_tol=0.0, what=f"{what} sparse q{i}")
        fusion_bit_exact(got, i, limit)
    n_pass = {}
    for i in range(B):
        f = None if fo[i] < 0 else fl[fo[i]]
        if int(fo[i]) not in n_pass:
            n_pass[int(fo[i])] = int(passes(w, f, np.arange(w["n"])).sum())
        for br in ("dense", "sparse"):
            hits = got.branch(i, br)
            rows = [r for r, _ in hits]
            sc = [s for _, s in hits]
            assert len(set(rows)) == len(rows), f"{what} {br} q{i}: duplicate rows"
            assert all(sc[t] >= sc[t + 1] for t in range(len(sc) - 1)), f"{what} {br} q{i}: not sorted"
            assert passes(w, f, rows).all(), f"{what} {br} q{i}: a row fails the query's filter or is deleted"
        assert len(got.branch(i, "dense")) == min(3 * limit, n_pass[int(fo[i])]), f"{what} q{i}: short list"


def assignment(B, count):
    """filter_of for `count` distinct filters: the first tile of 256 queries holds 256 distinct filters (a full tile
    table); later queries cycle through the rest, every 13th one unfiltered."""
    fo = (np.arange(B) % count).astype(np.int32)
    fo[256:][np.arange(256, B) % 13 == 5] = -1
    return fo


@pytest.mark.parametrize("count", [64, 256, 257, 1024])
def test_k2t_distinct_filters_per_query(big, count):
    w, eng = big, big["engine"]
    fl = distinct_filters(count, seed=count)
    fo = assignment(w["B"], count)
    got = w["ix"].search_batch(w["Q"], w["SP"], [eng.Filter(*f) for f in fl], fo, limit=100, fusion="rrf", branches=True)
    st = w["ix"].stats()
    assert st["last_dense_path"] == 2 and st["last_dense_passes"] == 1, st
    check_batch(w, got, fl, fo, f"K2T {count} filters")


def test_resident_k2_sub_batches_with_1024_filters(big):
    w, eng = big, big["engine"]
    fl = distinct_filters(1024, seed=4)
    fo = assignment(w["B"], 1024)
    w["ix"].set_option("k2_tiled", 0)
    try:
        got = w["ix"].search_batch(w["Q"], w["SP"], [eng.Filter(*f) for f in fl], fo, limit=100, fusion="rrf", branches=True)
        st = w["ix"].stats()
    finally:
        w["ix"].set_option("k2_tiled", 1)
    assert st["last_dense_path"] == 2 and st["last_dense_passes"] > 1, st
    check_batch(w, got, fl, fo, "resident K2 1024 filters")


def same(a, b):
    return all(np.array_equal(getattr(a, k), getattr(b, k)) for k in
               ("rows", "scores", "counts", "dense_rows", "dense_scores", "dense_counts", "sparse_rows", "sparse_scores", "sparse_counts"))


def test_content_equal_and_unused_filters_are_merged(big):
    w, eng, ix = big, big["engine"], big["ix"]
    B = w["B"]
    bits = np.zeros(2, np.uint32); bits[0] = np.uint32(0x0F0F3C5A)               # a scope-only filter, 16 of the 64 scopes
    shared = eng.Filter(bits, 0, 0, 0)
    # equal content, distinct objects: trailing zero words and the range of a filter without a date field do not count
    copies = [eng.Filter(np.concatenate([bits, np.zeros(i % 3, np.uint32)]), 0, -i, i * 7) for i in range(B)]
    ix.set_option("dense_compact", 70)
    ix.set_option("dense_compact_min_rows", 1024)
    try:
        one = ix.search_batch(w["Q"], w["SP"], [shared], np.zeros(B, np.int32), limit=100, fusion="rrf", branches=True)
        many = ix.search_batch(w["Q"], w["SP"], copies, np.arange(B, dtype=np.int32), limit=100, fusion="rrf", branches=True)
        assert ix.stats()["last_sel_used"] == 1, ix.stats()
    finally:
        ix.set_option("dense_compact", -1)
        ix.set_option("dense_compact_min_rows", 1 << 18)
    assert same(many, one)
    # 300 filters passed, 5 used: the unused ones are dropped
    fl = distinct_filters(300, seed=9)
    used = [3, 77, 150, 222, 299]
    fo = np.array([used[i % 5] for i in range(B)], np.int32)
    got = ix.search_batch(w["Q"], w["SP"], [eng.Filter(*f) for f in fl], fo, limit=100, fusion="rrf", branches=True)
    want = ix.search_batch(w["Q"], w["SP"], [eng.Filter(*fl[u]) for u in used], (np.arange(B) % 5).astype(np.int32),
                           limit=100, fusion="rrf", branches=True)
    assert same(got, want)


def test_two_shards_with_300_per_query_filters_equal_single_index(big):
    """vb_search_local on two row shards + vb_merge_fuse, as the multi-GPU layer runs them, with a distinct filter for
    most of 300 queries: the merged lists equal the single-index answer."""
    import torch
    w, eng = big, big["engine"]
    n, dim, half = w["n"], w["dim"], 70_016
    B, limit = 300, 20
    Q = w["Q"][:B]
    fl = distinct_filters(260, seed=11)
    fo = (np.arange(B) % 260).astype(np.int32); fo[::17] = -1
    gf = [eng.Filter(*f) for f in fl]
    shards = [eng.Index(dim, row_base=0), eng.Index(dim, row_base=half)]
    for hx, (lo, hi) in zip(shards, ((0, half), (half, n))):
        hx.upsert(w["dense"][lo:hi], None, w["scope"][lo:hi], None, w["modified"][lo:hi])
        dead = np.flatnonzero(~w["alive"][lo:hi])
        hx.delete_rows(dead + lo)                               # global row ids (row_base + local)
    try:
        want = w["ix"].search_batch(Q, None, gf, fo, limit=limit, fusion="dense", branches=True)
        words = eng.Index.cand_block_words(B, limit)
        gathered = torch.zeros(2 * words, dtype=torch.int64, device="cuda")
        for r, hx in enumerate(shards):
            hx.search_local(gathered[r * words:].data_ptr(), Q, None, gf, fo, limit=limit, kprime=limit, fusion="dense")
            assert hx.stats()["last_dense_path"] == 2
        torch.cuda.synchronize()
        merged = shards[0].merge_fuse(gathered.data_ptr(), 2, Q, None, limit=limit, kprime=limit, fusion="dense", branches=True)
        for i in range(B):
            assert merged.branch(i, "dense") == want.branch(i, "dense"), f"sharded per-query filters q{i}"
            assert merged.hits(i) == want.hits(i)
        assert any(r >= half for i in range(B) for r, _ in merged.branch(i, "dense"))
    finally:
        for hx in shards:
            hx.close()


def test_vector_store_search_batch_with_per_query_filters(monkeypatch):
    """The drop-in class: 300 queries, each with its own folder scope and date range, in one device batch (K2T) against
    one search() per query (single-query path) — same hits within the 1e-3 tolerance of the bf16 query operand."""
    from voitta_rag_b200 import vector_store as VS
    name = "gpu_per_query_filters"
    n, dim = 12_000, 64
    monkeypatch.setenv("QDRANT_COLLECTION", name)
    monkeypatch.setenv("EMBEDDING_DIMENSION", str(dim))
    VS._drop_collection(name)
    try:
        store = VS.VectorStoreService()
        corpus = _data.make_corpus(seed=17, n=n, dim=dim, n_index=6, per_index=6, vocab=2000)
        chunks = [(corpus["texts"][r], corpus["dense"][r].astype(float).tolist(), VS.ChunkMetadata(**corpus["metas"][r]))
                  for r in range(n)]
        store.store_chunks(chunks, [corpus["sparse"][r] for r in range(n)])
        folders = sorted({m["folder_path"] for m in corpus["metas"]})
        rng = np.random.RandomState(3)
        qs = _data.make_queries(seed=6, corpus=corpus, nq=300)
        filters = []
        for i in range(len(qs)):
            if i % 10 == 7:
                filters.append(None)
                continue
            kw = {"include_folders": sorted(rng.choice(folders, size=rng.randint(2, 30), replace=False).tolist())}
            if rng.rand() < 0.7:
                lo = T0 + int(rng.randint(0, 200_000_000))
                kw.update(date_start=lo, date_end=lo + int(rng.randint(30_000_000, 150_000_000)),
                          date_field=["created", "modified"][i % 2])
            filters.append(kw)
        Q = np.stack([q for q, _ in qs])
        got = store.search_batch(Q, limit=10, filters=filters)
        assert store.client.stats()["last_dense_path"] == 2
        for i in range(len(qs)):
            want = store.search(Q[i].astype(float).tolist(), limit=10, **(filters[i] or {}))
            assert_same_ranking([(c.id, c.score) for c in got[i]], [(c.id, c.score) for c in want],
                                rel_tol=1e-3, abs_tol=1e-3, what=f"drop-in q{i}")
    finally:
        VS._drop_collection(name)
