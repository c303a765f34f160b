"""GPU parity tests proper: the CUDA path (through the C ABI) against the oracle on identical
seeded inputs.  Tolerances: inputs are bf16-representable, so the fp32 paths (K1 dense scan,
K3 sparse, K4 fusion) must agree with the oracle to fp32 summation error (1e-5); the
tensor-core path (K2) feeds the unit query as bf16 hi+lo halves (bf16x2) when the batch fits one
pass and must then agree to 2e-5; with a plain bf16 query (k2_precision=1, throughput mode for
large batches) it is held to the north_star's stated 1e-3 relative tie tolerance."""
import math

import numpy as np
import pytest

import _data
import _coded
from _parity import assert_same_list, assert_same_ranking, assert_topk_valid
from oracle import oracle as O
from oracle import oracle_c

pytestmark = pytest.mark.gpu

FZ = {"weighted": 1, "rrf": 2}


def make_index(coded, dim, **opts):
    from voitta_rag_b200 import engine
    ix = engine.Index(dim)
    ix.upsert(coded["dense"], coded["csr"], coded["scope"], coded["created"], coded["modified"])
    for k, v in opts.items():
        ix.set_option(k, v)
    return ix


@pytest.fixture(scope="module")
def world():
    from voitta_rag_b200 import engine
    n, dim = 20000, 64
    corpus = _data.make_corpus(seed=3, n=n, dim=dim, n_index=6, per_index=6, vocab=3000)
    corpus["dense"][100] = corpus["dense"][99]          # exact tie
    corpus["sparse"][100] = corpus["sparse"][99]
    corpus["dense"][5] = 0.0
    queries = _data.make_queries(seed=9, corpus=corpus, nq=12)
    coded = _coded.code_corpus(corpus)
    cc = oracle_c.CorpusC(coded["dense"], coded["csr"], coded["scope"], coded["created"], coded["modified"])
    ix = make_index(coded, dim)
    return dict(n=n, dim=dim, corpus=corpus, queries=queries, coded=coded, cc=cc, ix=ix, engine=engine)


def filters_for(coded):
    sl = coded["scope_list"]
    folders = [f for f, _ in sl]
    return [
        None,
        (_coded.scope_bits(sl, include=folders[:5]), 0, _coded.TS_MIN, _coded.TS_MAX),
        (_coded.scope_bits(sl, exclude=folders[:2], disabled=["root3"]), 0, _coded.TS_MIN, _coded.TS_MAX),
        (None, 2, 1500000000, 1650000000),
        (_coded.scope_bits(sl, include=folders[3:20]), 1, 1450000000, _coded.TS_MAX),
        (_coded.scope_bits(sl, include=[folders[-1]]), 2, 1766000000, 1767225600),   # ~nothing passes
    ]


def run_both(w, qs, flt, limit, fusion, sparse_weight=0.1, use_sparse=True, **kw):
    eng = w["engine"]
    Q = np.stack([q for q, _ in qs])
    SP = [s for _, s in qs] if use_sparse else None
    B = len(qs)
    gf = None if flt is None else [eng.Filter(flt[0], flt[1], flt[2], flt[3])]
    fo = None if flt is None else np.zeros(B, np.int32)
    got = w["ix"].search_batch(Q, SP, gf, fo, limit=limit, fusion=fusion if use_sparse else "dense",
                               sparse_weight=sparse_weight, branches=True, **kw)
    want = w["cc"].search_batch(Q, SP, None if flt is None else [flt], fo, limit=limit,
                                kprime=got.dense_rows.shape[1],
                                fusion=FZ[fusion] if use_sparse else 0, sparse_weight=sparse_weight)
    return got, want


def check(got, want, B, tol, what):
    for i in range(B):
        gd = got.branch(i, "dense")
        wd = [(int(want["dense_rows"][i, j]), float(want["dense_scores"][i, j])) for j in range(want["dense_counts"][i])]
        assert_same_ranking(gd, wd, rel_tol=tol, abs_tol=tol, what=f"{what} dense q{i}")
        gs = got.branch(i, "sparse")
        ws = [(int(want["sparse_rows"][i, j]), float(want["sparse_scores"][i, j])) for j in range(want["sparse_counts"][i])]
        assert_same_list(gs, ws, what=f"{what} sparse q{i}")      # fp64 ordered sums: bit-equal
        gf = got.hits(i)
        wf = [(int(want["rows"][i, j]), float(want["scores"][i, j])) for j in range(want["counts"][i])]
        assert_same_ranking(gf, wf, rel_tol=10 * tol, abs_tol=10 * tol, what=f"{what} fused q{i}")


def fusion_bit_exact(got, i, limit, fusion, w):
    """K4 against the Python oracle's fusion, fed the GPU's own branch lists: ids, order and
    fp64 scores must be identical."""
    d = [O.ScoredPoint(str(r), s, {}, r) for r, s in got.branch(i, "dense")]
    s = [O.ScoredPoint(str(r), sc, {}, r) for r, sc in got.branch(i, "sparse")]
    if fusion == "rrf":
        want = O.reciprocal_rank_fusion([d, s], limit)
    else:
        want = O.weighted_fusion(d, s, limit, w)
    assert [(int(pid), sc) for pid, sc, _ in want] == got.hits(i)


@pytest.mark.parametrize("fusion", ["weighted", "rrf"])
@pytest.mark.parametrize("fi", range(6))
def test_single_query_hybrid_filtered(world, fusion, fi):
    flt = filters_for(world["coded"])[fi]
    for qi in range(6):
        got, want = run_both(world, world["queries"][qi:qi + 1], flt, 10, fusion, 0.3)
        check(got, want, 1, 1e-5, f"{fusion} f{fi} q{qi}")
        fusion_bit_exact(got, 0, 10, fusion, 0.3)
    assert world["ix"].stats()["last_dense_path"] == 3          # K1F: single query, small corpus


def test_dense_only_and_limits(world):
    for limit in (1, 10, 100, 341):
        for path, tol in ((1, 1e-5), (2, 2e-5)):
            world["ix"].set_option("dense_path", path)
            got, want = run_both(world, world["queries"][:3], None, limit, "weighted", use_sparse=False)
            for i in range(3):
                wf = [(int(want["rows"][i, j]), float(want["scores"][i, j])) for j in range(want["counts"][i])]
                assert_same_ranking(got.hits(i), wf, rel_tol=tol, abs_tol=tol, what=f"limit {limit} path {path}")
    world["ix"].set_option("dense_path", 0)


def test_weights_and_spread_zero(world):
    world["ix"].set_option("dense_path", 1)      # strict fp32 comparison below
    for w_sparse in (0.0, 0.5, 1.0):
        got, want = run_both(world, world["queries"][:4], None, 5, "weighted", w_sparse)
        check(got, want, 4, 1e-5, f"w={w_sparse}")
        for i in range(4):
            fusion_bit_exact(got, i, 5, "weighted", w_sparse)
    # a single sparse hit => spread == 0 => normalised score 1.0 (vector_store.py:667)
    corpus = world["corpus"]
    df = {}
    for idx, _ in corpus["sparse"]:
        for t in idx:
            df[t] = df.get(t, 0) + 1
    t1 = next(t for t, c in sorted(df.items()) if c == 1)
    q = world["queries"][0][0]
    got, want = run_both(world, [(q, ([t1], [1.0]))], None, 10, "weighted", 0.4)
    assert got.sparse_counts[0] == 1
    check(got, want, 1, 1e-5, "single sparse hit")
    fusion_bit_exact(got, 0, 10, "weighted", 0.4)
    # absent term => empty sparse list
    got, want = run_both(world, [(q, ([2**31 - 7], [1.0]))], None, 10, "rrf")
    assert got.sparse_counts[0] == 0
    check(got, want, 1, 1e-5, "absent term")
    world["ix"].set_option("dense_path", 0)


@pytest.mark.parametrize("path,prec", [(1, 0), (2, 0), (2, 1), (2, 2)])
def test_batch_paths(world, path, prec):
    """B = 12 through the GEMV scan (K1, one pass per query) and the tcgen05 GEMM (K2) with a
    bf16x2 (auto / forced) or plain bf16 query."""
    ix = world["ix"]
    ix.set_option("dense_path", path)
    ix.set_option("k2_precision", prec)
    try:
        tol = 1e-5 if path == 1 else (1e-3 if prec == 1 else 2e-5)
        for fi in (0, 1, 3):
            flt = filters_for(world["coded"])[fi]
            got, want = run_both(world, world["queries"], flt, 10, "rrf")
            assert ix.stats()["last_dense_path"] == path
            B = len(world["queries"])
            for i in range(B):
                gd = got.branch(i, "dense")
                wd = [(int(want["dense_rows"][i, j]), float(want["dense_scores"][i, j])) for j in range(want["dense_counts"][i])]
                assert_same_ranking(gd, wd, rel_tol=tol, abs_tol=tol, what=f"path {path} f{fi} dense q{i}")
                fusion_bit_exact(got, i, 10, "rrf", 0.1)
    finally:
        ix.set_option("dense_path", 0)
        ix.set_option("k2_precision", 0)


def test_per_query_filters_in_one_batch(world):
    eng = world["engine"]
    fl = [f for f in filters_for(world["coded"]) if f is not None]
    qs = world["queries"][:10]
    Q = np.stack([q for q, _ in qs])
    SP = [s for _, s in qs]
    fo = np.array([i % (len(fl) + 1) - 1 for i in range(len(qs))], np.int32)    # -1 = unfiltered
    for path in (1, 2):
        world["ix"].set_option("dense_path", path)
        got = world["ix"].search_batch(Q, SP, [eng.Filter(*f) for f in fl], fo, limit=10, fusion="weighted", branches=True)
        want = world["cc"].search_batch(Q, SP, fl, fo, limit=10, kprime=30, fusion=1)
        tol = 1e-5 if path == 1 else 2e-5
        for i in range(len(qs)):
            wd = [(int(want["dense_rows"][i, j]), float(want["dense_scores"][i, j])) for j in range(want["dense_counts"][i])]
            assert_same_ranking(got.branch(i, "dense"), wd, rel_tol=tol, abs_tol=tol, what=f"path{path} q{i}")
            ws = [(int(want["sparse_rows"][i, j]), float(want["sparse_scores"][i, j])) for j in range(want["sparse_counts"][i])]
            assert_same_list(got.branch(i, "sparse"), ws, what=f"path{path} sparse q{i}")
    world["ix"].set_option("dense_path", 0)


def test_segmentation_does_not_change_results(world):
    """Exactness is independent of the segment schedule (and of the safe mode)."""
    ix = world["ix"]
    qs = world["queries"][:6]
    Q = np.stack([q for q, _ in qs]); SP = [s for _, s in qs]
    base = ix.search_batch(Q, SP, limit=20, fusion="weighted", branches=True)
    try:
        for opts in ({"seg_ratio": 2}, {"seg_first": 16384, "seg_ratio": 2}, {"safe_mode": 1}):
            for k, v in opts.items():
                ix.set_option(k, v)
            r = ix.search_batch(Q, SP, limit=20, fusion="weighted", branches=True)
            for name in ("rows", "scores", "counts", "dense_rows", "dense_scores", "sparse_rows", "sparse_scores"):
                assert np.array_equal(getattr(r, name), getattr(base, name)), (opts, name)
            ix.set_option("safe_mode", 0); ix.set_option("seg_first", 2048); ix.set_option("seg_ratio", 0)
    finally:
        ix.set_option("safe_mode", 0); ix.set_option("seg_first", 2048); ix.set_option("seg_ratio", 0)


def test_deletes_update_mask_n_and_df(world):
    coded, dim = world["coded"], world["dim"]
    ix = make_index(coded, dim, dense_path=1)
    rng = np.random.RandomState(1)
    dead = rng.choice(world["n"], size=3000, replace=False)
    ix.delete_rows(dead)
    alive = np.ones(world["n"], np.uint8); alive[dead] = 0
    cc = oracle_c.CorpusC(coded["dense"], coded["csr"], coded["scope"], coded["created"], coded["modified"], alive)
    df, n_live = ix.term_stats(np.array([t for t in world["queries"][0][1][0]], np.uint32))
    assert n_live == world["n"] - 3000
    for t, d in zip(world["queries"][0][1][0], df):
        assert cc.df(t) == int(d)
    w2 = dict(world, ix=ix, cc=cc)
    for fi in (0, 1):
        got, want = run_both(w2, world["queries"][:5], filters_for(coded)[fi], 10, "weighted")
        check(got, want, 5, 1e-5, f"after delete f{fi}")
        assert not (set(int(r) for r in got.rows.ravel()) & set(int(x) for x in dead)) or got.counts.sum() == 0
    # append after delete, search again
    ix.upsert(coded["dense"][:500], (coded["csr"][0][:501], coded["csr"][1][:coded["csr"][0][500]], coded["csr"][2][:coded["csr"][0][500]]),
              coded["scope"][:500], coded["created"][:500], coded["modified"][:500])
    assert ix.stats()["n_rows"] == world["n"] + 500 and ix.stats()["n_live"] == world["n"] - 3000 + 500
    ix.close()


def test_overflow_falls_back_to_safe_mode_and_stays_exact():
    """Adversarial order (scores strictly increasing with the row id) floods the candidate lists;
    the library must notice, re-run in safe mode and still return the exact answer."""
    from voitta_rag_b200 import engine
    n, dim = 700000, 64          # (tiny batches get 262144-slot lists: the corpus must outgrow them)
    theta = np.linspace(1.5, 0.05, n).astype(np.float64)
    dense = np.zeros((n, dim), np.float32)
    dense[:, 0] = np.cos(theta); dense[:, 1] = np.sin(theta)
    dense = _data.bf16_round(dense)
    ix = engine.Index(dim)
    ix.upsert(dense)
    q = np.zeros(dim, np.float32); q[0] = 1.0
    v = dense.astype(np.float64)
    scores = (v[:, 0] / np.linalg.norm(v, axis=1)).astype(np.float32)
    # the single-pass scan (K1F) keeps its candidates in per-CTA buffers that it re-selects as often as needed: no overflow
    ix.set_option("k1f", 2)        # (2 = also on corpora larger than the 2M rows K1F is used for by default)
    r = ix.search_batch(q[None, :], limit=10)
    assert ix.stats()["overflow_reruns"] == 0
    assert_topk_valid(r.hits(0), scores, np.ones(n, bool), 10, rel_tol=1e-6, abs_tol=1e-6, what="ascending corpus, K1F")
    # the segmented kernels (here K1 with k1f = 0; batches use the same lists) overflow, notice, and re-run in safe mode
    ix.set_option("k1f", 0)
    r = ix.search_batch(q[None, :], limit=10)
    assert ix.stats()["overflow_reruns"] == 1
    assert_topk_valid(r.hits(0), scores, np.ones(n, bool), 10, rel_tol=1e-6, abs_tol=1e-6, what="ascending corpus")
    # and a batch on the tensor-core path
    r = ix.search_batch(np.stack([q, q, q]), limit=10)
    assert ix.stats()["overflow_reruns"] == 2
    for i in range(3):
        assert_topk_valid(r.hits(i), scores, np.ones(n, bool), 10, rel_tol=1e-3, abs_tol=1e-3, what="ascending corpus, K2")
    ix.close()


@pytest.mark.parametrize("dim", [100, 384, 768, 1024, 1536])
def test_dimensions_and_padding(dim):
    from voitta_rag_b200 import engine
    rng = np.random.RandomState(dim)
    n = 4000
    dense = _data.bf16_round(rng.randn(n, dim).astype(np.float32))
    Q = _data.bf16_round(rng.randn(5, dim).astype(np.float32))
    ix = engine.Index(dim)
    ix.upsert(dense)
    cc = oracle_c.CorpusC(dense)
    want = cc.search_batch(Q, None, limit=10, fusion=0)
    for path, tol in ((1, 1e-5), (2, 2e-5)):
        ix.set_option("dense_path", path)
        got = ix.search_batch(Q, limit=10)
        for i in range(5):
            wf = [(int(want["rows"][i, j]), float(want["scores"][i, j])) for j in range(want["counts"][i])]
            assert_same_ranking(got.hits(i), wf, rel_tol=tol, abs_tol=tol, what=f"dim {dim} path {path} q{i}")
    ix.close()


def test_two_shards_merge_equals_single_index(world):
    """Row-sharded search (SURVEY §8e) emulated on one GPU: two indexes with row offsets, global
    IDF from summed df, candidates concatenated as an all-gather would, merged and fused.  Must be
    bit-identical to the single-index answer."""
    import torch
    eng, coded, dim, n = world["engine"], world["coded"], world["dim"], world["n"]
    half = 8192 + 1000
    ip, tm, vl = coded["csr"]
    a = eng.Index(dim, row_base=0)
    a.upsert(coded["dense"][:half], (ip[:half + 1], tm[:ip[half]], vl[:ip[half]]), coded["scope"][:half],
             coded["created"][:half], coded["modified"][:half])
    b = eng.Index(dim, row_base=half)
    b.upsert(coded["dense"][half:], (ip[half:] - ip[half], tm[ip[half]:], vl[ip[half]:]), coded["scope"][half:],
             coded["created"][half:], coded["modified"][half:])
    qs = world["queries"][:8]
    Q = np.stack([q for q, _ in qs]); SP = [s for _, s in qs]
    flt = filters_for(coded)[1]
    gf, fo = [eng.Filter(*flt)], np.zeros(len(qs), np.int32)
    # global IDF: df summed over shards, N = total live
    SPW = []
    for idx, val in SP:
        t = np.asarray(idx, np.uint32)
        dfa, na = a.term_stats(t); dfb, nb = b.term_stats(t)
        N = na + nb
        wts = [float(v) * math.log((N - float(d) + 0.5) / (float(d) + 0.5) + 1.0) for v, d in zip(val, (dfa + dfb))]
        SPW.append((idx, wts))
    limit, k = 10, 30
    for fusion in ("weighted", "rrf"):
        single = world["ix"].search_batch(Q, SP, gf, fo, limit=limit, fusion=fusion, branches=True)
        bufs = [torch.zeros(eng.Index.cand_block_words(len(qs), k), dtype=torch.int64, device="cuda") for _ in range(2)]
        a.search_local(bufs[0].data_ptr(), Q, SPW, gf, fo, limit=limit, kprime=k, fusion=fusion)
        b.search_local(bufs[1].data_ptr(), Q, SPW, gf, fo, limit=limit, kprime=k, fusion=fusion)
        gathered = torch.cat(bufs)
        torch.cuda.synchronize()
        merged = a.merge_fuse(gathered.data_ptr(), 2, Q, SPW, limit=limit, kprime=k, fusion=fusion, branches=True)
        for name in ("rows", "counts", "dense_rows", "dense_scores", "dense_counts", "sparse_rows", "sparse_counts"):
            assert np.array_equal(getattr(merged, name), getattr(single, name)), (fusion, name)
        # idf computed by numpy here vs libm in the library may differ in the last bit of a weight
        np.testing.assert_allclose(merged.sparse_scores, single.sparse_scores, rtol=1e-6)
        # the same with the threshold exchange of the sharded flow (all-reduce MAX emulated with torch.maximum):
        # shards keep fewer candidates, the merged answer is identical
        taus = []
        staged = []
        for sh_ix in (a, b):
            staged.append(sh_ix.stage(Q, SPW, gf, fo, limit=limit, kprime=k, fusion=fusion, apply_idf=False, branches=True))
            sh_ix.run_local_begin()
            t = torch.zeros(2 * len(qs), dtype=torch.float32, device="cuda")
            sh_ix.tau_export(t.data_ptr())
            taus.append(t)
        torch.cuda.synchronize()
        tmax = torch.maximum(taus[0], taus[1])
        torch.cuda.synchronize()
        for sh_ix, buf in zip((a, b), bufs):
            sh_ix.tau_import(tmax.data_ptr())
            sh_ix.run_local(buf.data_ptr())
        torch.cuda.synchronize()
        gathered2 = torch.cat(bufs)
        a.run_fuse(2, gathered2.data_ptr())
        shared = a.fetch(staged[0])
        for name in ("rows", "counts", "dense_rows", "dense_scores", "dense_counts", "sparse_rows", "sparse_counts"):
            assert np.array_equal(getattr(shared, name), getattr(merged, name)), ("threshold exchange", fusion, name)
        assert np.array_equal(shared.sparse_scores, merged.sparse_scores)
        np.testing.assert_allclose(merged.scores, single.scores, rtol=1e-6, atol=1e-9)
    a.close(); b.close()


def test_upsert_dev_matches_host_upsert(world):
    import torch
    eng, coded, dim = world["engine"], world["coded"], world["dim"]
    n = 9000
    ip, tm, vl = coded["csr"]
    rows = torch.from_numpy(coded["dense"][:n]).cuda().to(torch.bfloat16).contiguous()
    t_ip = torch.from_numpy(ip[:n + 1].copy()).cuda(); t_tm = torch.from_numpy(tm[:ip[n]].astype(np.int32)).cuda()
    t_vl = torch.from_numpy(vl[:ip[n]].copy()).cuda()
    t_sc = torch.from_numpy(coded["scope"][:n].astype(np.int32)).cuda()
    t_cr = torch.from_numpy(coded["created"][:n].copy()).cuda(); t_mo = torch.from_numpy(coded["modified"][:n].copy()).cuda()
    torch.cuda.synchronize()
    d = eng.Index(dim)
    d.upsert_dev(n, rows.data_ptr(), t_ip.data_ptr(), t_tm.data_ptr(), t_vl.data_ptr(), t_sc.data_ptr(),
                 t_cr.data_ptr(), t_mo.data_ptr())
    h = eng.Index(dim)
    h.upsert(coded["dense"][:n], (ip[:n + 1], tm[:ip[n]], vl[:ip[n]]), coded["scope"][:n], coded["created"][:n], coded["modified"][:n])
    qs = world["queries"][:4]
    Q = np.stack([q for q, _ in qs]); SP = [s for _, s in qs]
    flt = filters_for(coded)[4]
    ra = d.search_batch(Q, SP, [eng.Filter(*flt)], np.zeros(4, np.int32), limit=10, fusion="rrf", branches=True)
    rb = h.search_batch(Q, SP, [eng.Filter(*flt)], np.zeros(4, np.int32), limit=10, fusion="rrf", branches=True)
    for name in ("rows", "scores", "counts", "dense_rows", "dense_scores", "sparse_rows", "sparse_scores"):
        assert np.array_equal(getattr(ra, name), getattr(rb, name)), name
    d.close(); h.close()


def test_edge_cases(world):
    eng = world["engine"]
    e = eng.Index(16)
    r = e.search_batch(np.ones((2, 16), np.float32), limit=5)
    assert r.counts.tolist() == [0, 0]                                  # empty index
    e.upsert(np.eye(16, dtype=np.float32)[:3])                          # fewer rows than k
    r = e.search_batch(np.ones((1, 16), np.float32), [([1, 2], [1.0, 1.0])], limit=5, fusion="rrf", branches=True)
    assert r.counts[0] == 3 and r.sparse_counts[0] == 0
    with pytest.raises(ValueError):
        e.search_batch(np.full((1, 16), np.nan, np.float32))
    with pytest.raises(eng.B200Error):
        e.search_batch(np.ones((1, 16), np.float32), limit=400, kprime=1200)
    with pytest.raises(eng.B200Error):
        e.search_batch(np.ones((1, 16), np.float32), [([3, 3], [1.0, 1.0])], limit=5)   # repeated sparse index
    with pytest.raises(eng.B200Error):
        e.delete_rows([99])
    e.close()


def test_large_batch_hybrid_against_oracle():
    """BASELINE cfg2 shape scaled down (300k x 128, B = 64, hybrid RRF + weighted): exercises the
    tcgen05 path with several segments, the sub-range append counters, the two-stream schedule and
    the pipelined stream API; checked row by row against the C oracle."""
    from voitta_rag_b200 import engine
    rng = np.random.RandomState(5)
    n, dim, B = 300_000, 128, 64
    cents = rng.randn(512, dim).astype(np.float32)
    dense = cents[rng.randint(0, 512, size=n)] + 0.5 * rng.randn(n, dim).astype(np.float32)
    dense = _data.bf16_round(dense)
    # sparse rows: 12 terms from a Zipf vocabulary of 20k hashed ids
    vocab = np.unique(rng.randint(1, 2**31 - 1, size=40000).astype(np.int64))[:20000]
    p = 1.0 / np.arange(1, len(vocab) + 1) ** 1.07
    p /= p.sum()
    L = 12
    picks = rng.choice(len(vocab), size=(n, L), p=p)
    picks.sort(axis=1)
    keep = np.ones((n, L), bool); keep[:, 1:] = picks[:, 1:] != picks[:, :-1]
    terms_sorted_ids = np.argsort(np.argsort(vocab))            # rank of each vocab entry by hashed id
    hashed = np.sort(vocab)
    rows_terms = [np.unique(hashed[terms_sorted_ids[picks[r][keep[r]]]]) for r in range(n)]
    indptr = np.zeros(n + 1, np.int64); np.cumsum([len(t) for t in rows_terms], out=indptr[1:])
    terms = np.concatenate(rows_terms).astype(np.uint32)
    vals = (1.0 + rng.rand(len(terms))).astype(np.float32)
    scope = rng.randint(0, 64, size=n).astype(np.uint32)
    modified = rng.randint(1420070400, 1767225600, size=n).astype(np.int64)
    ix = engine.Index(dim)
    ix.upsert(dense, (indptr, terms, vals), scope, None, modified)
    cc = oracle_c.CorpusC(dense, (indptr, terms, vals), scope, None, modified)
    qrows = rng.randint(0, n, size=B)
    Q = _data.bf16_round(dense[qrows] + 0.3 * rng.randn(B, dim).astype(np.float32))
    SP = [(rows_terms[r][:6].tolist() + [int(hashed[rng.randint(0, len(hashed))])], [1.0] * 7) for r in qrows]
    SP = [(list(dict.fromkeys(t)), [1.0] * len(dict.fromkeys(t))) for t, _ in SP]
    bits = np.zeros(2, np.uint32); bits[0] = 0x0F0F0F0F; bits[1] = 0xFFFF0000
    flt = (bits, 2, 1500000000, 1767225600)
    fo = np.zeros(B, np.int32)
    for fusion, fz in (("rrf", 2), ("weighted", 1)):
        got = ix.search_batch(Q, SP, [engine.Filter(*flt)], fo, limit=10, fusion=fusion, branches=True)
        assert ix.stats()["last_dense_path"] == 2
        want = cc.search_batch(Q, SP, [flt], fo, limit=10, fusion=fz)
        for i in range(B):
            wd = [(int(want["dense_rows"][i, j]), float(want["dense_scores"][i, j])) for j in range(want["dense_counts"][i])]
            assert_same_ranking(got.branch(i, "dense"), wd, rel_tol=2e-5, abs_tol=2e-5, what=f"dense q{i}")
            ws = [(int(want["sparse_rows"][i, j]), float(want["sparse_scores"][i, j])) for j in range(want["sparse_counts"][i])]
            assert_same_list(got.branch(i, "sparse"), ws, what=f"sparse q{i}")
            fusion_bit_exact(got, i, 10, fusion, 0.1)
    # MaxScore pruning forced on: identical sparse lists (bit for bit) and fused results
    base = ix.search_batch(Q, SP, [engine.Filter(*flt)], fo, limit=10, fusion="rrf", branches=True)
    ix.set_option("sparse_prune_force", 1)
    pruned = ix.search_batch(Q, SP, [engine.Filter(*flt)], fo, limit=10, fusion="rrf", branches=True)
    ix.set_option("sparse_prune_force", 0)
    for i in range(B):
        assert pruned.branch(i, "sparse") == base.branch(i, "sparse"), f"pruned sparse list q{i}"
        assert pruned.hits(i) == base.hits(i)
    # relaxed mode (dense columns for frequent terms, order-free sums + verification) against exact mode
    # (sparse_dense = 0: every term walked in term order): identical lists, bit for bit
    assert ix.stats()["n_terms"] > 0
    ix.set_option("sparse_dense", 0)
    exact = ix.search_batch(Q, SP, [engine.Filter(*flt)], fo, limit=10, fusion="rrf", branches=True)
    ix.set_option("sparse_dense", 1)
    for i in range(B):
        assert exact.branch(i, "sparse") == base.branch(i, "sparse"), f"exact vs relaxed sparse list q{i}"
    # query values of either sign and zero: such queries always take the exact mode; still bit-equal to the oracle
    SPm = [(t, [float(v) for v in rng.choice([-1.0, 0.0, 0.5, 1.0, 2.0], size=len(t))]) for t, _ in SP]
    gotm = ix.search_batch(Q, SPm, [engine.Filter(*flt)], fo, limit=10, fusion="rrf", branches=True)
    wantm = cc.search_batch(Q, SPm, [flt], fo, limit=10, fusion=2)
    for i in range(B):
        ws = [(int(wantm["sparse_rows"][i, j]), float(wantm["sparse_scores"][i, j])) for j in range(wantm["sparse_counts"][i])]
        assert_same_list(gotm.branch(i, "sparse"), ws, what=f"mixed-sign sparse q{i}")
    # the pipelined stream API returns the same answers as the one-call API
    packed = [ix.pack(Q[j:j + 16], SP[j:j + 16], [engine.Filter(*flt)], np.zeros(16, np.int32), limit=10, fusion="rrf")
              for j in range(0, B, 16)]
    one = [ix.search_batch(Q[j:j + 16], SP[j:j + 16], [engine.Filter(*flt)], np.zeros(16, np.int32), limit=10, fusion="rrf")
           for j in range(0, B, 16)]
    for a, b in zip(ix.search_stream(iter(packed)), one):
        assert np.array_equal(a.rows, b.rows) and np.array_equal(a.scores, b.scores) and np.array_equal(a.counts, b.counts)
    ix.close()


@pytest.mark.parametrize("budget", [20, 100])
def test_maxscore_pruning_is_exact(world, budget):
    """MaxScore pruning of the sparse branch (non-essential terms skipped, survivors re-scored from the
    forward index) forced on for every segment: the sparse lists stay bit-identical to the oracle's
    ordered fp64 sums, with and without filters, and with a tighter (20 %) or the full (100 %) budget."""
    ix = world["ix"]
    ix.set_option("sparse_prune_force", 1)
    ix.set_option("sparse_prune", budget)
    ix.set_option("seg_ratio", 4)                       # more segments => thresholds (and plans) change more often
    try:
        for fi in (0, 1, 3, 5):
            flt = filters_for(world["coded"])[fi]
            for limit in (10, 40):
                got, want = run_both(world, world["queries"], flt, limit, "weighted")
                check(got, want, len(world["queries"]), 1e-5, f"prune {budget}% f{fi} limit {limit}")
    finally:
        ix.set_option("sparse_prune_force", 0)
        ix.set_option("sparse_prune", 20)
        ix.set_option("seg_ratio", 0)


def test_query_tiled_gemm_large_batch():
    """B = 600 > the resident sub-batch: the query-tiled tcgen05 kernel (256-query tiles, the last one
    partial) against the C oracle at the north_star's 1e-3 relative tie tolerance (plain bf16 query),
    and bit-identical to the multi-pass resident kernel, for every mask mode of the epilogue:
    no filter, one filter for the whole batch, a few filters, and more than 31 filters."""
    from voitta_rag_b200 import engine
    rng = np.random.RandomState(11)
    n, dim, B = 80_000, 128, 600
    cents = rng.randn(256, dim).astype(np.float32)
    dense = _data.bf16_round(cents[rng.randint(0, 256, size=n)] + 0.6 * rng.randn(n, dim).astype(np.float32))
    scope = rng.randint(0, 64, size=n).astype(np.uint32)
    modified = rng.randint(1420070400, 1767225600, size=n).astype(np.int64)
    ix = engine.Index(dim)
    ix.upsert(dense, None, scope, None, modified)
    cc = oracle_c.CorpusC(dense, None, scope, None, modified)
    Q = _data.bf16_round(dense[rng.randint(0, n, size=B)] + 0.4 * rng.randn(B, dim).astype(np.float32))
    bits = np.zeros(2, np.uint32); bits[0] = 0x00FFFF00; bits[1] = 0x0F0F0F0F
    span = 1767225600 - 1420070400
    few = [(bits, 0, 0, 0), (None, 2, 1500000000, 1700000000), (bits, 2, 1450000000, 1767225600)]
    many = [(None, 2, 1420070400 + i * span // 80, 1420070400 + (i + 40) * span // 80) for i in range(40)]
    cases = [
        ("none", None, None),
        ("uniform", few[:1], np.zeros(B, np.int32)),
        ("few", few, (np.arange(B) % 4 - 1).astype(np.int32)),
        ("many", many, (np.arange(B) % 41 - 1).astype(np.int32)),
    ]
    try:
        for name, fl, fo in cases:
            filters = None if fl is None else [engine.Filter(*f) for f in fl]
            ix.set_option("k2_tiled", 1)
            got = ix.search_batch(Q, None, filters, fo, limit=10, fusion="dense")
            st = ix.stats()
            assert st["last_dense_path"] == 2 and st["last_dense_passes"] == 1, st
            ix.set_option("k2_tiled", 0)
            ref = ix.search_batch(Q, None, filters, fo, limit=10, fusion="dense")
            assert ix.stats()["last_dense_passes"] > 1
            assert np.array_equal(got.counts, ref.counts), name
            for i in range(B):
                assert got.hits(i) == ref.hits(i), f"tiled vs resident kernel, {name} q{i}"
            want = cc.search_batch(Q, None, fl, fo, limit=10, fusion=0)
            for i in range(B):
                wf = [(int(want["rows"][i, j]), float(want["scores"][i, j])) for j in range(want["counts"][i])]
                assert_same_ranking(got.hits(i), wf, rel_tol=1e-3, abs_tol=1e-3, what=f"tiled {name} q{i}")
    finally:
        ix.close()


def test_snapshot_save_load_roundtrip(world, tmp_path):
    """vb_save / vb_load: the restored shard (rows, columns, tombstones, forward CSR; inverted index
    rebuilt) answers hybrid filtered searches bit-identically, deletes included."""
    eng = world["engine"]
    coded = world["coded"]
    ix = make_index(coded, world["dim"])
    ix.delete_rows([7, 99, 1234])
    qs = world["queries"]
    Q = np.stack([q for q, _ in qs]); SP = [s for _, s in qs]
    flt = filters_for(coded)[4]
    args = dict(filters=[eng.Filter(*flt)], filter_of=np.zeros(len(qs), np.int32), limit=10, fusion="weighted", branches=True)
    want = ix.search_batch(Q, SP, **args)
    path = tmp_path / "shard.vb200"
    ix.save(path)
    st = ix.stats()
    ix.close()
    jx = eng.Index.load(path, device=0)
    try:
        s2 = jx.stats()
        assert (jx.dim, s2["n_rows"], s2["n_live"], s2["nnz"]) == (world["dim"], st["n_rows"], st["n_live"], st["nnz"])
        got = jx.search_batch(Q, SP, **args)
        for i in range(len(qs)):
            assert got.hits(i) == want.hits(i)
            assert got.branch(i, "dense") == want.branch(i, "dense") and got.branch(i, "sparse") == want.branch(i, "sparse")
        # the restored index keeps accepting writes
        first = jx.upsert(coded["dense"][:5], (coded["csr"][0][:6] - coded["csr"][0][0], coded["csr"][1][:coded["csr"][0][5]], coded["csr"][2][:coded["csr"][0][5]]),
                          coded["scope"][:5], coded["created"][:5], coded["modified"][:5])
        assert first == st["n_rows"] and jx.stats()["n_live"] == st["n_live"] + 5
    finally:
        jx.close()
    with pytest.raises(eng.B200Error):
        eng.Index.load(tmp_path / "missing.vb200")


def test_full_size_cfg2_properties():
    """BASELINE configs[1] at FULL size (1M x 384, batch 64, top-10 hybrid RRF) through size-independent
    properties (the oracle comparison at this size is bench.py's parity_spot_check):
      * the sparse branch of a query does not depend on the batch it travels in (B = 64 vs B = 1), bit for bit;
      * the dense branch agrees between the tensor-core batch path and the single-query scan within the stated
        1e-3 tie tolerance;
      * top-10 is a prefix of top-20 for both branches;
      * splitting the corpus into two shards and merging (the multi-GPU flow, emulated on one GPU) gives the
        single-index answer; deleting a query's best row removes exactly that row from its lists."""
    import torch
    from voitta_rag_b200 import engine, synth
    dev = torch.device("cuda", 0)
    n, dim, B = 1_000_000, 384, 64
    ix = engine.Index(dim)
    halves = [engine.Index(dim, row_base=0), engine.Index(dim, row_base=n // 2)]
    keep = None
    for blk in range(n // 125_000):
        rows = synth.dense_rows(125_000, dim, blk, dev, "C")
        ip, tm, vl = synth.sparse_rows(125_000, blk, dev)
        sc, cr, mo = synth.columns(125_000, blk, dev)
        torch.cuda.synchronize()
        for target in (ix, halves[0] if blk < 4 else halves[1]):
            target.upsert_dev(125_000, rows.data_ptr(), ip.data_ptr(), tm.data_ptr(), vl.data_ptr(), sc.data_ptr(),
                              cr.data_ptr(), mo.data_ptr())
        if keep is None:
            keep = (rows, ip, tm)
    Q, SP = synth.queries(B, 0, keep[0], keep[1], keep[2])
    try:
        full = ix.search_batch(Q, SP, limit=10, fusion="rrf", branches=True)
        assert ix.stats()["last_dense_path"] == 2
        wide = ix.search_batch(Q, SP, limit=20, kprime=60, fusion="rrf", branches=True)
        for i in range(B):
            assert len(full.branch(i, "dense")) == 30 and len(full.hits(i)) == 10
            assert wide.branch(i, "sparse")[:30] == full.branch(i, "sparse"), f"sparse prefix q{i}"
            assert_same_ranking(wide.branch(i, "dense")[:30], full.branch(i, "dense"), rel_tol=1e-6, abs_tol=1e-6, what=f"dense prefix q{i}")
        for i in (0, 17, 63):
            one = ix.search_batch(Q[i:i + 1], SP[i:i + 1], limit=10, fusion="rrf", branches=True)
            assert ix.stats()["last_dense_path"] in (1, 3)      # K1 (corpus > 2M rows) or K1F
            assert one.branch(0, "sparse") == full.branch(i, "sparse"), f"sparse batch independence q{i}"
            assert_same_ranking(full.branch(i, "dense"), one.branch(0, "dense"), rel_tol=1e-3, abs_tol=1e-3, what=f"K2 vs K1 q{i}")
        # two shards + merge == one index (global idf: weights computed once from the full index)
        terms = np.asarray(sorted({int(t) for s in SP for t in s[0]}), np.uint32)
        df, n_live = ix.term_stats(terms)
        dfm = dict(zip(terms.tolist(), df.tolist()))
        W = [(s[0], [v * math.log((n_live - dfm[t] + 0.5) / (dfm[t] + 0.5) + 1.0) for t, v in zip(s[0], s[1])]) for s in SP]
        words = engine.Index.cand_block_words(B, 30)
        gathered = torch.zeros(2 * words, dtype=torch.int64, device=dev)
        for r, hx in enumerate(halves):
            hx.search_local(gathered[r * words:].data_ptr(), Q, W, None, None, limit=10, kprime=30, fusion="rrf")
        torch.cuda.synchronize()
        merged = halves[0].merge_fuse(gathered.data_ptr(), 2, Q, W, limit=10, kprime=30, fusion="rrf", branches=True)
        for i in range(B):
            assert merged.branch(i, "sparse") == full.branch(i, "sparse"), f"sharded sparse q{i}"
            assert merged.branch(i, "dense") == full.branch(i, "dense"), f"sharded dense q{i}"
            assert merged.hits(i) == full.hits(i)
        # delete the best dense row of query 0: it disappears, everything else keeps its order
        best = full.branch(0, "dense")[0][0]
        ix.delete_rows([best])
        after = ix.search_batch(Q[:1], SP[:1], limit=10, fusion="rrf", branches=True)
        assert best not in [r for r, _ in after.branch(0, "dense")] and best not in [r for r, _ in after.branch(0, "sparse")]
    finally:
        ix.close()
        for hx in halves:
            hx.close()


@pytest.mark.parametrize("seed", [1, 2])
def test_sparse_relaxed_mode_stress(seed):
    """Relaxed sparse mode under stress: a small vocabulary (dozens of dense columns, queries that hold many of
    them), queries of 1 .. 256 terms (the term table spans several 32-term chunks), posting values that are zero,
    denormal, tiny and huge in the same corpus, weights over 30 orders of magnitude — sparse lists must equal the
    oracle's ordered fp64 sums bit for bit, through several segments, with and without a filter."""
    from voitta_rag_b200 import engine
    rng = np.random.RandomState(100 + seed)
    n, dim, V = 20_000, 32, 400
    dense = _data.bf16_round(rng.randn(n, dim).astype(np.float32))
    vocab = np.unique(rng.randint(1, 2**31 - 1, size=4 * V).astype(np.int64))[:V]      # sorted, distinct
    assert len(vocab) == V
    p = 1.0 / np.arange(1, V + 1) ** 0.9
    p /= p.sum()
    lens = rng.randint(20, 121, size=n)
    picks = rng.choice(V, size=(n, 120), p=p)
    picks[np.arange(120)[None, :] >= lens[:, None]] = V          # beyond the row's length: sentinel, sorted last
    picks.sort(axis=1)
    keep = np.ones_like(picks, bool)
    keep[:, 1:] = picks[:, 1:] != picks[:, :-1]
    keep &= picks < V
    counts = keep.sum(axis=1)
    indptr = np.zeros(n + 1, np.int64); np.cumsum(counts, out=indptr[1:])
    terms = vocab[picks[keep]].astype(np.uint32)                  # row-major, ascending (vocab is sorted)
    nnz = len(terms)
    kind = rng.randint(0, 10, size=nnz)
    vals = (0.2 + 2.0 * rng.rand(nnz)).astype(np.float32)
    vals[kind == 0] = 0.0
    vals[kind == 1] = np.float32(1e-42)          # denormal
    vals[kind == 2] = np.float32(3e-30)
    vals[kind == 3] = np.float32(7e18)
    scope = rng.randint(0, 8, size=n).astype(np.uint32)
    ix = engine.Index(dim)
    ix.upsert(dense, (indptr, terms, vals), scope, None, None)
    cc = oracle_c.CorpusC(dense, (indptr, terms, vals), scope, None, None)
    nts = [1, 2, 5, 31, 32, 33, 64, 100, 200, 256, 7, 12]
    SP = []
    for nt in nts:
        t = np.sort(rng.choice(V, size=min(nt, V), replace=False))
        w = (10.0 ** rng.uniform(-15, 15, size=len(t))) if nt % 2 else (0.5 + rng.rand(len(t)))
        SP.append((vocab[t].tolist(), [float(x) for x in w]))
    B = len(SP)
    Q = _data.bf16_round(rng.randn(B, dim).astype(np.float32))
    bits = np.zeros(1, np.uint32); bits[0] = 0b10110101
    try:
        ix.set_option("seg_ratio", 4)
        for apply_idf in (True, False):
            for fl, fo in ((None, None), ([(bits, 0, 0, 0)], np.zeros(B, np.int32))):
                filters = None if fl is None else [engine.Filter(*f) for f in fl]
                got = ix.search_batch(Q, SP, filters, fo, limit=20, fusion="rrf", branches=True, apply_idf=apply_idf)
                want = cc.search_batch(Q, SP, fl, fo, limit=20, fusion=2, apply_idf=apply_idf)
                for i in range(B):
                    ws = [(int(want["sparse_rows"][i, j]), float(want["sparse_scores"][i, j])) for j in range(want["sparse_counts"][i])]
                    assert_same_list(got.branch(i, "sparse"), ws, what=f"stress nt={nts[i]} idf={apply_idf} filter={fl is not None}")
        assert ix.stats()["overflow_reruns"] <= 8
    finally:
        ix.close()


def test_k3m_equals_k3_and_oracle(world):
    """The posting-driven MaxScore kernel (K3M, sparse_ms.cuh) and the block x query kernel (K3) must return
    the same sparse lists bit for bit — under every filter, budget, work-unit size and segment schedule —
    and both equal the oracle's ordered fp64 sums."""
    ix, coded = world["ix"], world["coded"]
    qs = world["queries"]
    Q = np.stack([q for q, _ in qs]); SP = [s for _, s in qs]
    B = len(qs)
    eng = world["engine"]
    try:
        for fi, flt in enumerate(filters_for(coded)):
            gf = None if flt is None else [eng.Filter(*flt)]
            fo = None if flt is None else np.zeros(B, np.int32)
            ix.set_option("sparse_ms", 0)
            base = ix.search_batch(Q, SP, gf, fo, limit=20, fusion="rrf", branches=True)
            ix.set_option("sparse_ms", 1)
            for opts in ({}, {"ms_chunk": 512}, {"ms_chunk": 8192, "ms_budget": 20}, {"ms_budget": 0},
                         {"seg_ratio": 2}, {"seg_first": 16384, "seg_ratio": 2, "ms_chunk": 512}, {"safe_mode": 1},
                         {"sparse_dense": 0}):
                for k, v in opts.items():
                    ix.set_option(k, v)
                r = ix.search_batch(Q, SP, gf, fo, limit=20, fusion="rrf", branches=True)
                for name in ("rows", "scores", "counts", "sparse_rows", "sparse_scores", "sparse_counts"):
                    assert np.array_equal(getattr(r, name), getattr(base, name)), (fi, opts, name)
                for k in opts:
                    ix.set_option(k, {"ms_chunk": 0, "ms_budget": 100, "seg_ratio": 0, "seg_first": 2048, "safe_mode": 0, "sparse_dense": 1}[k])
            want = world["cc"].search_batch(Q, SP, None if flt is None else [flt], fo, limit=20, kprime=60, fusion=2)
            for i in range(B):
                ws = [(int(want["sparse_rows"][i, j]), float(want["sparse_scores"][i, j])) for j in range(want["sparse_counts"][i])]
                assert_same_list(base.branch(i, "sparse"), ws, what=f"k3m f{fi} q{i}")
    finally:
        for k, v in {"sparse_ms": 1, "ms_chunk": 0, "ms_budget": 100, "seg_ratio": 0, "seg_first": 2048, "safe_mode": 0, "sparse_dense": 1}.items():
            ix.set_option(k, v)


def _csr_slice(csr, lo, hi):
    ip, tm, vl = csr
    return (ip[lo:hi + 1] - ip[lo], tm[ip[lo]:ip[hi]], vl[ip[lo]:ip[hi]])


def test_incremental_upserts_and_deletes_interleaved(world):
    """The reference interleaves store_chunks batches of 100 and per-file deletes with searches
    (indexing.py:434,560,284).  Writes must not rebuild the inverted index: appended rows are scored as a delta
    from the forward index, deletes only clear alive bits, N and df follow both.  After EVERY write the hybrid
    results (every filter shape, both kernels' paths) are compared with the oracle on the same live set."""
    from voitta_rag_b200 import engine
    coded, dim, n = world["coded"], world["dim"], world["n"]
    qs = world["queries"][:6]
    Q = np.stack([q for q, _ in qs]); SP = [s for _, s in qs]
    B = len(qs)
    n0 = 12000
    ix = engine.Index(dim)
    ix.upsert(coded["dense"][:n0], _csr_slice(coded["csr"], 0, n0), coded["scope"][:n0], coded["created"][:n0], coded["modified"][:n0])
    alive = np.ones(n, np.uint8)
    rng = np.random.RandomState(7)
    flts = filters_for(coded)

    def compare(rows_now, what):
        cc = oracle_c.CorpusC(coded["dense"][:rows_now], _csr_slice(coded["csr"], 0, rows_now), coded["scope"][:rows_now],
                              coded["created"][:rows_now], coded["modified"][:rows_now], alive[:rows_now])
        for t in SP[0][0]:
            df, n_live = ix.term_stats(np.array([t], np.uint32))
            assert int(df[0]) == cc.df(t) and n_live == int(alive[:rows_now].sum()), (what, t)
        for fi in (0, 1, 3):
            flt = flts[fi]
            gf = None if flt is None else [engine.Filter(*flt)]
            fo = None if flt is None else np.zeros(B, np.int32)
            for path in (1, 2):
                ix.set_option("dense_path", path)
                got = ix.search_batch(Q, SP, gf, fo, limit=10, fusion="weighted", branches=True)
                want = cc.search_batch(Q, SP, None if flt is None else [flt], fo, limit=10, kprime=30, fusion=1)
                check(got, want, B, 1e-5 if path == 1 else 2e-5, f"{what} f{fi} path{path}")
        ix.set_option("dense_path", 0)

    compare(n0, "initial")
    assert ix.stats()["index_builds"] == 1
    rows_now = n0
    for step in range(8):
        if step % 2 == 0:                                   # a store_chunks batch
            add = 100
            ix.upsert(coded["dense"][rows_now:rows_now + add], _csr_slice(coded["csr"], rows_now, rows_now + add),
                      coded["scope"][rows_now:rows_now + add], coded["created"][rows_now:rows_now + add], coded["modified"][rows_now:rows_now + add])
            rows_now += add
        else:                                               # delete a few "files" (3 consecutive chunks), old and new rows
            starts = rng.randint(0, rows_now - 3, size=5)
            dead = np.unique(np.concatenate([np.arange(s0, s0 + 3) for s0 in starts]))
            ix.delete_rows(dead.astype(np.uint64))
            alive[dead] = 0
        compare(rows_now, f"step{step}")
        st = ix.stats()
        assert st["index_builds"] == 1 and st["delta_rows"] == rows_now - n0, st
    # a query term that exists only in the delta rows: df comes from the adjustment table alone
    new_term = int(coded["csr"][1].max()) + 17
    extra = np.zeros((2, dim), np.float32); extra[:, 0] = 1.0
    ix.upsert(extra, (np.array([0, 1, 2], np.int64), np.array([new_term, new_term], np.uint32), np.array([1.5, 0.5], np.float32)),
              np.zeros(2, np.uint32), None, None)
    got = ix.search_batch(Q[:1], [([new_term], [1.0])], limit=5, fusion="rrf", branches=True)
    assert got.branch(0, "sparse")[0][0] == rows_now and got.sparse_counts[0] == 2
    idf = math.log((int(alive[:rows_now].sum()) + 2 - 2 + 0.5) / (2 + 0.5) + 1.0)
    assert got.branch(0, "sparse")[0][1] == float(np.float32(idf * 1.5))
    ix.delete_rows(np.array([rows_now, rows_now + 1], np.uint64))
    # crossing the threshold merges the delta inside vb_upsert (off the search path); results unchanged
    ix.set_option("delta_max", 400)
    alive2 = np.concatenate([alive[:rows_now], np.zeros(2, np.uint8)])
    add = 200
    ix.upsert(coded["dense"][rows_now:rows_now + add], _csr_slice(coded["csr"], rows_now, rows_now + add),
              coded["scope"][rows_now:rows_now + add], coded["created"][rows_now:rows_now + add], coded["modified"][rows_now:rows_now + add])
    st = ix.stats()
    assert st["index_builds"] == 2 and st["delta_rows"] == 0, st
    # rows rows_now, rows_now+1 are the two deleted extras: the oracle corpus skips them via its alive mask
    dense2 = np.concatenate([coded["dense"][:rows_now], extra, coded["dense"][rows_now:rows_now + add]])
    def cat_csr(a, b):
        return (np.concatenate([a[0], a[0][-1] + b[0][1:]]), np.concatenate([a[1], b[1]]), np.concatenate([a[2], b[2]]))
    csr2 = cat_csr(cat_csr(_csr_slice(coded["csr"], 0, rows_now), (np.array([0, 1, 2], np.int64), np.array([new_term, new_term], np.uint32), np.array([1.5, 0.5], np.float32))),
                   _csr_slice(coded["csr"], rows_now, rows_now + add))
    sc2 = np.concatenate([coded["scope"][:rows_now], np.zeros(2, np.uint32), coded["scope"][rows_now:rows_now + add]])
    cr2 = np.concatenate([coded["created"][:rows_now], np.full(2, _coded.TS_MISSING, np.int64), coded["created"][rows_now:rows_now + add]])
    mo2 = np.concatenate([coded["modified"][:rows_now], np.full(2, _coded.TS_MISSING, np.int64), coded["modified"][rows_now:rows_now + add]])
    al2 = np.concatenate([alive2, np.ones(add, np.uint8)])
    cc = oracle_c.CorpusC(dense2, csr2, sc2, cr2, mo2, al2)
    got = ix.search_batch(Q, SP, limit=10, fusion="weighted", branches=True)
    want = cc.search_batch(Q, SP, None, None, limit=10, kprime=30, fusion=1)
    check(got, want, B, 2e-5, "after merge")
    # vb_optimize with nothing to merge is a no-op; after a delete it rebuilds and drops the dead postings
    ix.optimize()
    assert ix.stats()["index_builds"] == 2
    ix.delete_rows(np.array([5, 6], np.uint64)); al2[[5, 6]] = 0
    ix.optimize()
    assert ix.stats()["index_builds"] == 3
    cc = oracle_c.CorpusC(dense2, csr2, sc2, cr2, mo2, al2)
    got = ix.search_batch(Q, SP, limit=10, fusion="weighted", branches=True)
    want = cc.search_batch(Q, SP, None, None, limit=10, kprime=30, fusion=1)
    check(got, want, B, 2e-5, "after optimize")
    ix.close()


@pytest.mark.parametrize("dim", [768, 1024])
def test_query_tiled_gemm_at_model_dimensions_against_oracle(dim):
    """K2T (the query-tiled tcgen05 kernel) at the dimensions the north_star names (768 = e5-base-v2, 1024), B = 1024,
    limit 100 (k' = 300), all four epilogue mask modes, hybrid on a corpus >> k'.  The oracle scores a 96-query
    subset per mode (the dense oracle is O(B x n x d) on the CPU); the other queries are held to the size-independent
    properties (sorted, unique rows, pass their filter)."""
    from voitta_rag_b200 import engine
    rng = np.random.RandomState(dim)
    n, B, limit = 150_000, 1024, 100
    cents = rng.randn(256, dim).astype(np.float32)
    dense = _data.bf16_round(cents[rng.randint(0, 256, size=n)] + 0.7 * rng.randn(n, dim).astype(np.float32))
    vocab = np.unique(rng.randint(1, 2**31 - 1, size=8000).astype(np.int64))[:4000]
    p = 1.0 / np.arange(1, len(vocab) + 1) ** 1.07; p /= p.sum()
    L = 10
    picks = np.sort(rng.choice(len(vocab), size=(n, L), p=p), axis=1)
    rows_terms = [np.unique(vocab[picks[r]]) for r in range(n)]
    indptr = np.zeros(n + 1, np.int64); np.cumsum([len(t) for t in rows_terms], out=indptr[1:])
    terms = np.concatenate(rows_terms).astype(np.uint32)
    vals = (0.5 + 1.5 * rng.rand(len(terms))).astype(np.float32)
    scope = rng.randint(0, 64, size=n).astype(np.uint32)
    modified = rng.randint(1420070400, 1767225600, size=n).astype(np.int64)
    ix = engine.Index(dim)
    ix.upsert(dense, (indptr, terms, vals), scope, None, modified)
    cc = oracle_c.CorpusC(dense, (indptr, terms, vals), scope, None, modified)
    qrows = rng.randint(0, n, size=B)
    Q = _data.bf16_round(dense[qrows] + 0.4 * rng.randn(B, dim).astype(np.float32))
    SP = [(list(dict.fromkeys(rows_terms[r][:5].tolist() + [int(vocab[rng.randint(0, len(vocab))])])), None) for r in qrows]
    SP = [(t, [1.0] * len(t)) for t, _ in SP]

    def flt(k):
        bits = np.zeros(2, np.uint32); bits[0] = np.uint32((0x9E3779B1 * (k + 1)) & 0xFFFFFFFF); bits[1] = np.uint32((0x85EBCA77 * (k + 3)) & 0xFFFFFFFF)
        return (bits, 2, 1420070400 + k * 1_000_000, 1767225600)
    modes = {"none": (None, None), "uniform": ([flt(0)], np.zeros(B, np.int32)),
             "few": ([flt(k) for k in range(8)], (np.arange(B) % 8).astype(np.int32)),
             "many": ([flt(k) for k in range(40)], (np.arange(B) % 40).astype(np.int32))}
    sub = np.sort(rng.choice(B, size=96, replace=False))
    coded = {"scope": scope, "created": None, "modified": modified}
    for name, (fl, fo) in modes.items():
        gf = None if fl is None else [engine.Filter(*f) for f in fl]
        got = ix.search_batch(Q, SP, gf, fo, limit=limit, fusion="rrf", branches=True)
        st = ix.stats()
        assert st["last_dense_path"] == 2 and st["last_dense_passes"] == 1, st          # one corpus pass for 1024 queries = K2T
        assert got.dense_rows.shape[1] == 300
        want = cc.search_batch(Q[sub], [SP[i] for i in sub], fl, None if fo is None else fo[sub], limit=limit, kprime=300, fusion=2)
        for j, i in enumerate(sub):
            wd = [(int(want["dense_rows"][j, t]), float(want["dense_scores"][j, t])) for t in range(want["dense_counts"][j])]
            assert_same_ranking(got.branch(i, "dense"), wd, rel_tol=1e-3, abs_tol=1e-3, what=f"K2T d{dim} {name} dense q{i}")
            ws = [(int(want["sparse_rows"][j, t]), float(want["sparse_scores"][j, t])) for t in range(want["sparse_counts"][j])]
            assert_same_list(got.branch(i, "sparse"), ws, what=f"K2T d{dim} {name} sparse q{i}")
            fusion_bit_exact(got, i, limit, "rrf", 0.1)
        for i in range(0, B, 37):                     # properties for queries the oracle did not score
            rows = [r for r, _ in got.branch(i, "dense")]
            sc = [s_ for _, s_ in got.branch(i, "dense")]
            assert len(set(rows)) == len(rows) and all(sc[t] >= sc[t + 1] for t in range(len(sc) - 1))
            if fl is not None:
                f = fl[int(fo[i])]
                ok = ((f[0][scope[rows] >> 5] >> (scope[rows] & 31)) & 1).astype(bool) & (modified[rows] >= f[2]) & (modified[rows] <= f[3])
                assert ok.all(), f"K2T d{dim} {name} q{i}: a returned row fails its filter"
    ix.close()


def test_k1f_single_pass_equals_segmented_scan_and_oracle(world):
    """K1F (one pass, per-CTA candidate buffers, thresholds shared through one global word) against K1 in row segments:
    identical lists for B = 1..8, every filter, limits up to 100 (k' = 300), exact ties included; and against the oracle."""
    ix, coded, eng = world["ix"], world["coded"], world["engine"]
    qs = world["queries"]
    ix.set_option("dense_path", 1)
    try:
        for B in (1, 3, 8):
            Q = np.stack([q for q, _ in qs[:B]]); SP = [s for _, s in qs[:B]]
            for fi, flt in enumerate(filters_for(coded)):
                gf = None if flt is None else [eng.Filter(*flt)]
                fo = None if flt is None else np.zeros(B, np.int32)
                for limit in (10, 100):
                    ix.set_option("k1f", 0)
                    base = ix.search_batch(Q, SP, gf, fo, limit=limit, fusion="weighted", branches=True)
                    ix.set_option("k1f", 1)
                    fast = ix.search_batch(Q, SP, gf, fo, limit=limit, fusion="weighted", branches=True)
                    for name in ("rows", "scores", "counts", "dense_rows", "dense_scores", "dense_counts", "sparse_rows", "sparse_scores", "sparse_counts"):
                        assert np.array_equal(getattr(fast, name), getattr(base, name)), (B, fi, limit, name)
            got, want = run_both(world, qs[:B], filters_for(coded)[1], 10, "rrf")
            check(got, want, B, 1e-5, f"k1f B{B}")
        # dense-only, duplicate rows (exact tie between rows 99 and 100) around the cut-off
        q = world["corpus"]["dense"][99][None, :]
        for k1f in (0, 1):
            ix.set_option("k1f", k1f)
            r = ix.search_batch(q, None, limit=2, fusion="dense", branches=True)
            assert [int(x) for x in r.rows[0, :2]] == [99, 100], (k1f, r.rows)
    finally:
        ix.set_option("k1f", 1); ix.set_option("dense_path", 0)


def test_k3h_long_queries_equal_k3_and_oracle(world):
    """Long queries (more than ms_max_terms terms) go to K3H, the hash-accumulate MaxScore kernel: the sparse lists must be
    bit-identical to K3's (sparse_mh = 0) and to the oracle's, in a batch that also holds short (K3M) and mixed-sign (K3)
    queries, under every filter, in safe mode and with a tiny ms_max_terms (every query long)."""
    ix, coded, eng = world["ix"], world["coded"], world["engine"]
    long_qs = _data.make_queries(seed=77, corpus=world["corpus"], nq=10, nnz=(17, 24))
    assert max(len(s[0]) for _, s in long_qs) > 16
    qs = long_qs + world["queries"][:4]
    Q = np.stack([q for q, _ in qs]); SP = [s for _, s in qs]
    SP[-1] = (SP[-1][0], [-1.0] + [1.0] * (len(SP[-1][0]) - 1))           # a query K3 must keep (negative weight)
    B = len(qs)
    try:
        for fi, flt in enumerate(filters_for(coded)):
            gf = None if flt is None else [eng.Filter(*flt)]
            fo = None if flt is None else np.zeros(B, np.int32)
            ix.set_option("sparse_mh", 0)
            base = ix.search_batch(Q, SP, gf, fo, limit=20, fusion="rrf", branches=True)
            ix.set_option("sparse_mh", 1)
            for opts in ({}, {"ms_max_terms": 2}, {"safe_mode": 1}, {"seg_ratio": 2}, {"ms_staged": 0}, {"sparse_dense": 0}):
                for k, v in opts.items():
                    ix.set_option(k, v)
                r = ix.search_batch(Q, SP, gf, fo, limit=20, fusion="rrf", branches=True)
                for name in ("rows", "scores", "counts", "sparse_rows", "sparse_scores", "sparse_counts"):
                    assert np.array_equal(getattr(r, name), getattr(base, name)), (fi, opts, name)
                for k in opts:
                    ix.set_option(k, {"ms_max_terms": 16, "safe_mode": 0, "seg_ratio": 0, "ms_staged": 1, "sparse_dense": 1}[k])
            want = world["cc"].search_batch(Q, SP, None if flt is None else [flt], fo, limit=20, kprime=60, fusion=2)
            for i in range(B):
                ws = [(int(want["sparse_rows"][i, j]), float(want["sparse_scores"][i, j])) for j in range(want["sparse_counts"][i])]
                assert_same_list(base.branch(i, "sparse"), ws, what=f"k3h f{fi} q{i}")
    finally:
        for k, v in {"sparse_mh": 0, "ms_max_terms": 16, "safe_mode": 0, "seg_ratio": 0, "ms_staged": 1, "sparse_dense": 1}.items():
            ix.set_option(k, v)


@pytest.mark.parametrize("B", [320, 40])
def test_k2t_row_selection_equals_in_place_scoring_and_oracle(B):
    """B = 320: K2T (query-tiled), B = 40: K2 (resident queries, bf16x2) — both over the compacted copy of the rows that pass a batch-wide filter (dense_compact.cuh) must return exactly
    what K2T returns with the filter bit tested in its epilogue (same operands, same accumulation: identical keys),
    and both must match the oracle.  Selectivities from nothing to everything, tombstones, rows appended after the
    index build, a row count that is not a multiple of the tile."""
    from voitta_rag_b200 import engine
    rng = np.random.RandomState(77)
    n, dim, limit = 61_003, 128, 10
    cents = rng.randn(64, dim).astype(np.float32)
    dense = _data.bf16_round(cents[rng.randint(0, 64, size=n)] + 0.6 * rng.randn(n, dim).astype(np.float32))
    scope = rng.randint(0, 100, size=n).astype(np.uint32)
    modified = rng.randint(1420070400, 1767225600, size=n).astype(np.int64)
    ix = engine.Index(dim)
    n0 = 50_000                                            # the rest arrives later: delta rows (dense covers them all)
    ix.upsert(dense[:n0], None, scope[:n0], None, modified[:n0])
    Q = _data.bf16_round(dense[rng.randint(0, n, size=B)] + 0.3 * rng.randn(B, dim).astype(np.float32))
    ix.search_batch(Q[:4], None, limit=3, fusion="dense")  # builds the index state before the append
    ix.upsert(dense[n0:], None, scope[n0:], None, modified[n0:])
    dead = rng.choice(n, size=900, replace=False)
    ix.delete_rows(dead)
    alive = np.ones(n, bool); alive[dead] = False
    cc = oracle_c.CorpusC(dense, None, scope, None, modified, alive=alive.astype(np.uint8))

    def scope_filter(ids, lo=1420070400, hi=1767225600):
        bits = np.zeros(4, np.uint32)
        for s in ids:
            bits[s >> 5] |= np.uint32(1 << (s & 31))
        return (bits, 2, lo, hi)
    cases = {"1 scope of 100": scope_filter([7]), "half": scope_filter(range(0, 100, 2)), "all": scope_filter(range(100)),
             "none": scope_filter([]), "60 % and a date range": scope_filter(range(60), 1500000000, 1700000000)}
    fo = np.zeros(B, np.int32)
    sub = np.sort(rng.choice(B, size=min(B, 48), replace=False))
    tol = 1e-3 if B > 256 else 2e-5                        # plain bf16 query (K2T) / bf16x2 query (resident K2)
    for name, f in cases.items():
        passing = ((f[0][scope >> 5] >> (scope & 31)) & 1).astype(bool) & (modified >= f[2]) & (modified <= f[3]) & alive
        res = {}
        for sel in (0, 70):
            ix.set_option("dense_compact", sel)
            ix.set_option("dense_compact_min_rows", 1024)
            res[sel] = ix.search_batch(Q, None, [engine.Filter(*f)], fo, limit=limit, fusion="dense", branches=True)
            st = ix.stats()
            assert st["last_dense_path"] == 2 and st["last_dense_passes"] == 1, st
            if sel:
                assert st["last_sel_rows"] > 0 or passing.sum() == 0 or name == "none", (name, st)
                big_share = st["last_sel_rows"] / max(1, st["last_big_rows"])
                assert st["last_sel_used"] == (1 if big_share <= 0.70 else 0), (name, st)
            else:
                assert st["last_sel_used"] == 0
        for i in range(B):
            assert res[70].branch(i, "dense") == res[0].branch(i, "dense"), f"row selection changed the answer: {name} q{i}"
            rows = [r for r, _ in res[70].branch(i, "dense")]
            assert passing[rows].all(), f"{name} q{i}: a returned row fails the filter or is deleted"
            assert len(rows) == min(limit, int(passing.sum()))
        want = cc.search_batch(Q[sub], None, [f], fo[sub], limit=limit, kprime=limit, fusion=0)
        for j, i in enumerate(sub):
            wd = [(int(want["dense_rows"][j, t]), float(want["dense_scores"][j, t])) for t in range(want["dense_counts"][j])]
            assert_same_ranking(res[70].branch(i, "dense"), wd, rel_tol=tol, abs_tol=tol, what=f"row selection B={B} {name} q{i}")
    # every query on the SECOND filter of the batch: its words start at mask + 1 * mask_words, and 61003 rows are 1907
    # words — not 16-byte aligned (the selection kernels must not assume it)
    ix.set_option("dense_compact", 70)
    two = ix.search_batch(Q, None, [engine.Filter(*cases["all"]), engine.Filter(*cases["half"])], np.ones(B, np.int32), limit=limit,
                          fusion="dense", branches=True)
    assert ix.stats()["last_sel_used"] == 1
    one = ix.search_batch(Q, None, [engine.Filter(*cases["half"])], fo, limit=limit, fusion="dense", branches=True)
    for i in range(B):
        assert two.branch(i, "dense") == one.branch(i, "dense"), f"second filter of two, q{i}"
    ix.close()


def test_full_size_cfg4_shard_properties():
    """BASELINE configs[3] at the FULL per-GPU size (12.5M x 768 bf16, batch 1024, top-100 => k' = 300, scope + time
    filter at 50 %) through properties that do not need an O(B x n x d) oracle pass:
      * every returned dense score is the cosine of THAT row (the row is regenerated from its seed and scored on the
        host in fp64) within the stated 1e-3; every returned row passes the filter (columns regenerated the same way);
      * the lists are sorted (score desc, row asc on ties) and free of duplicates;
      * no row of a random sample of passing rows beats a list's k'-th score by more than the tolerance (exhaustiveness);
      * the tensor-core kernel over the row selection's compacted copy returns exactly what it returns in place;
      * a query's sparse branch is the same, bit for bit, alone (B = 1) and inside the batch; its dense branch agrees
        between the fp32 scan (B = 1) and the bf16 tensor path within 1e-3."""
    import sys
    import torch
    from pathlib import Path
    root = str(Path(__file__).resolve().parents[1])
    if root not in sys.path:
        sys.path.insert(0, root)
    import bench
    from voitta_rag_b200 import engine, synth
    dev = torch.device("cuda", 0)
    cfg = dict(bench.WORKLOADS["cfg4"])
    B, limit, kprime, dim = cfg["batch"], cfg["limit"], 3 * cfg["limit"], cfg["dim"]
    ix, keep, (lo, hi), _ = bench.build_shard(cfg, 0, 1, dev, torch, synth, engine)
    try:
        batches, flt = bench.make_batches(cfg, keep, 1, synth, engine, torch)
        Q, SP = batches[0]
        fo = np.zeros(B, np.int32)
        F = [engine.Filter(*flt)]
        res = {}
        for sel in (0, -1):
            ix.set_option("dense_compact", sel)
            res[sel] = ix.search_batch(Q, SP, F, fo, limit=limit, fusion="rrf", branches=True)
            st = ix.stats()
            assert st["last_dense_path"] == 2 and st["last_dense_passes"] == 1
            assert st["last_sel_used"] == (1 if sel else 0), st
        got = res[-1]
        for i in range(B):
            assert got.branch(i, "dense") == res[0].branch(i, "dense"), f"row selection changed dense list {i}"
            assert got.hits(i) == res[0].hits(i)
        # regenerate the blocks that hold the rows of a few lists and score them on the host
        blocks = {}

        def block(blk):
            if blk not in blocks:
                if len(blocks) >= 6:
                    blocks.pop(next(iter(blocks)))
                rows = synth.dense_rows(bench.BLOCK_ROWS, dim, blk, dev, cfg["dist"])
                sc, cr, mo = synth.columns(bench.BLOCK_ROWS, blk, dev)
                blocks[blk] = (rows, sc, mo)
            return blocks[blk]

        bits = np.asarray(flt[0], np.uint32)

        def passes(sc, mo):
            return bool((int(bits[sc >> 5]) >> (sc & 31)) & 1) and flt[2] <= mo <= flt[3]

        rng = np.random.RandomState(5)
        for i in (0, 311, 1023):
            lst = got.branch(i, "dense")
            assert len(lst) == kprime
            keys = [(-s, r) for r, s in lst]
            assert keys == sorted(keys) and len({r for r, _ in lst}) == kprime, f"list {i} not sorted / not unique"
            q = torch.from_numpy(np.asarray(Q[i], np.float64)).to(dev)
            q = q / q.norm()
            by_block = {}
            for r, s in lst:
                by_block.setdefault(r // bench.BLOCK_ROWS, []).append((r, s))
            for blk, items in sorted(by_block.items())[:40]:
                rows, sc, mo = block(blk)
                idx = torch.tensor([r % bench.BLOCK_ROWS for r, _ in items], device=dev)
                x = rows[idx].double()
                cos = ((x @ q) / x.norm(dim=1)).cpu().numpy()
                scs, mos = sc[idx].cpu().numpy(), mo[idx].cpu().numpy()
                for (r, s), c, a, m in zip(items, cos, scs, mos):
                    assert abs(s - c) <= 1e-3 * max(1.0, abs(c)), f"list {i} row {r}: score {s} vs cosine {c}"
                    assert passes(int(a), int(m)), f"list {i} row {r} fails the filter"
            # exhaustiveness on a sample: passing rows of two random blocks must not beat the k'-th score
            kth = lst[-1][1]
            for blk in rng.choice(cfg["n"] // bench.BLOCK_ROWS, size=2, replace=False):
                rows, sc, mo = block(int(blk))
                x = rows.double()
                cos = (x @ q) / x.norm(dim=1)
                bw = torch.from_numpy(bits.astype(np.int64)).to(dev)
                ok = (((bw[(sc.long() >> 5)] >> (sc.long() & 31)) & 1) == 1) & (mo >= flt[2]) & (mo <= flt[3])
                best = float(torch.where(ok, cos, torch.full_like(cos, -2.0)).max())
                inlist = {r for r, _ in lst}
                top = int(torch.where(ok, cos, torch.full_like(cos, -2.0)).argmax()) + int(blk) * bench.BLOCK_ROWS
                assert best <= kth + 1e-3 or top in inlist, f"list {i}: row {top} ({best}) beats the k'-th score {kth} but is missing"
        for i in (0, 1023):
            one = ix.search_batch(Q[i:i + 1], SP[i:i + 1], F, fo[:1], limit=limit, fusion="rrf", branches=True)
            assert ix.stats()["last_dense_path"] in (1, 3)
            assert one.branch(0, "sparse") == got.branch(i, "sparse"), f"sparse batch independence q{i}"
            assert_same_ranking(got.branch(i, "dense"), one.branch(0, "dense"), rel_tol=1e-3, abs_tol=1e-3, what=f"K2T vs K1 q{i}")
    finally:
        ix.close()


def test_row_selection_in_the_sharded_flow():
    """Two row shards (row_base 0 / n/2) under one batch-wide filter, tensor-core path over each shard's compacted copy,
    candidates merged as the multi-GPU layer does (vb_search_local x 2 -> vb_merge_fuse): the dense lists must equal
    the single-index answer — a candidate's id is row_base + the shard row the selection recorded."""
    import torch
    from voitta_rag_b200 import engine
    rng = np.random.RandomState(91)
    n, dim, B, limit = 40_000, 128, 320, 10
    dense = _data.bf16_round(rng.randn(n, dim).astype(np.float32))
    scope = rng.randint(0, 64, size=n).astype(np.uint32)
    modified = rng.randint(1420070400, 1767225600, size=n).astype(np.int64)
    Q = _data.bf16_round(dense[rng.randint(0, n, size=B)] + 0.3 * rng.randn(B, dim).astype(np.float32))
    bits = np.zeros(2, np.uint32); bits[0] = np.uint32(0x0F0F3C5A); bits[1] = np.uint32(0x00FF0011)
    flt = engine.Filter(bits, 2, 1450000000, 1767225600)
    fo = np.zeros(B, np.int32)
    one = engine.Index(dim)
    one.upsert(dense, None, scope, None, modified)
    halves = [engine.Index(dim, row_base=0), engine.Index(dim, row_base=n // 2)]
    halves[0].upsert(dense[:n // 2], None, scope[:n // 2], None, modified[:n // 2])
    halves[1].upsert(dense[n // 2:], None, scope[n // 2:], None, modified[n // 2:])
    try:
        for ix in [one] + halves:
            ix.set_option("dense_compact", 100)
            ix.set_option("dense_compact_min_rows", 1024)
        want = one.search_batch(Q, None, [flt], fo, limit=limit, fusion="dense", branches=True)
        assert one.stats()["last_sel_used"] == 1
        words = engine.Index.cand_block_words(B, limit)
        dev = torch.device("cuda", 0)
        gathered = torch.zeros(2 * words, dtype=torch.int64, device=dev)
        for r, hx in enumerate(halves):
            hx.search_local(gathered[r * words:].data_ptr(), Q, None, [flt], fo, limit=limit, kprime=limit, fusion="dense")
            assert hx.stats()["last_sel_used"] == 1
        torch.cuda.synchronize()
        merged = halves[0].merge_fuse(gathered.data_ptr(), 2, Q, None, limit=limit, kprime=limit, fusion="dense", branches=True)
        for i in range(B):
            assert merged.branch(i, "dense") == want.branch(i, "dense"), f"sharded row selection q{i}"
            assert merged.hits(i) == want.hits(i)
        assert any(r >= n // 2 for i in range(B) for r, _ in merged.branch(i, "dense"))
    finally:
        one.close()
        for hx in halves:
            hx.close()
