"""The C restatement (oracle/oracle_c.c) must agree with the line-cited Python oracle."""
import numpy as np
import pytest

import _data
import _coded
from _parity import assert_same_list, assert_same_ranking
from oracle import oracle as O
from oracle import oracle_c


@pytest.fixture(scope="module")
def setup():
    corpus = _data.make_corpus(seed=11, n=1500, dim=48, n_index=4, per_index=5)
    corpus["dense"][7] = 0.0
    queries = _data.make_queries(seed=5, corpus=corpus, nq=8)
    store = O.OracleVectorStore(48)
    ids = [f"{r:08d}" for r in range(1500)]
    store.store_chunks([(corpus["texts"][r], corpus["dense"][r].tolist(), O.ChunkMetadata(**corpus["metas"][r]))
                        for r in range(1500)], corpus["sparse"], ids=ids)
    coded = _coded.code_corpus(corpus)
    cc = oracle_c.CorpusC(coded["dense"], coded["csr"], coded["scope"], coded["created"], coded["modified"])
    return corpus, queries, store, coded, cc


CASES = [
    dict(),
    dict(include_folders=["root0", "root1/sub0", "root2"]),
    dict(exclude_folders=["root0"], exclude_index_folders=["root3"]),
    dict(date_start=1500000000, date_end=1700000000),
    dict(date_start=1500000000, date_field="created", include_folders=["root0", "root1", "root2", "root3"]),
]


@pytest.mark.parametrize("case", range(len(CASES)))
@pytest.mark.parametrize("fusion", ["weighted", "rrf"])
def test_c_oracle_matches_python_oracle(setup, case, fusion):
    corpus, queries, store, coded, cc = setup
    kw = CASES[case]
    store.fusion = fusion
    bits = _coded.scope_bits(coded["scope_list"], None, kw.get("include_folders"), kw.get("exclude_folders"),
                             kw.get("exclude_index_folders"))
    field = 0
    if "date_start" in kw or "date_end" in kw:
        field = 1 if kw.get("date_field") == "created" else 2
    flt = (bits, field, kw.get("date_start", _coded.TS_MIN), kw.get("date_end", _coded.TS_MAX))
    use_filter = bits is not None or field
    out = cc.search_batch(np.stack([q for q, _ in queries]), [s for _, s in queries],
                          filters=[flt] if use_filter else None,
                          filter_of=np.zeros(len(queries), np.int32) if use_filter else None,
                          limit=10, fusion={"weighted": 1, "rrf": 2}[fusion], sparse_weight=0.3)
    for i, (q, sq) in enumerate(queries):
        want = store.search(q.tolist(), limit=10, sparse_query=sq, sparse_weight=0.3, **kw)
        got = [(f"{int(out['rows'][i, j]):08d}", out["scores"][i, j]) for j in range(out["counts"][i])]
        assert_same_ranking(got, [(c.id, c.score) for c in want], rel_tol=2e-6, abs_tol=2e-6, what=f"q{i} {kw} {fusion}")
        flt_o = O.build_filter(None, kw.get("include_folders"), kw.get("exclude_folders"),
                               kw.get("exclude_index_folders"), kw.get("date_start"), kw.get("date_end"),
                               kw.get("date_field"))
        d, s = store.search_branches(q.tolist(), 10, flt_o, sq)
        gd = [(int(out["dense_rows"][i, j]), out["dense_scores"][i, j]) for j in range(out["dense_counts"][i])]
        gs = [(int(out["sparse_rows"][i, j]), out["sparse_scores"][i, j]) for j in range(out["sparse_counts"][i])]
        assert_same_ranking(gd, [(p.row, p.score) for p in d], rel_tol=2e-6, abs_tol=1e-7, what=f"dense q{i}")
        # sparse scores: identical arithmetic (f64 accumulate in index order) -> bit-equal
        assert_same_list(gs, [(p.row, p.score) for p in s], what=f"sparse q{i}")


def test_dense_only_and_df(setup):
    corpus, queries, store, coded, cc = setup
    out = cc.search_batch(np.stack([q for q, _ in queries]), None, limit=7, fusion=0)
    for i, (q, _) in enumerate(queries):
        want = store.search(q.tolist(), limit=7)
        got = [(f"{int(out['rows'][i, j]):08d}", out["scores"][i, j]) for j in range(out["counts"][i])]
        assert_same_ranking(got, [(c.id, c.score) for c in want], rel_tol=2e-6, abs_tol=1e-7)
    for t in list(store.coll.df)[:50]:
        assert cc.df(t) == store.coll.df[t]
