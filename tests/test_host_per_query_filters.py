"""Per-query filters through the host layer on a CPU box: VectorStoreService.search_batch(filters=[...]) against one
search() per query, its argument errors, and a two-rank sharded batch with hundreds of per-query filters against the
unsharded answer.  The index is the C-oracle test double; the GPU side of the feature is
tests/test_gpu_per_query_filters.py."""
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import _coded
import _data
from golden import make_golden as G
from _fake_index import FakeIndex
from oracle import oracle_c
from test_sharded_gloo import FakeShardIndex
from voitta_rag_b200 import engine
from voitta_rag_b200 import vector_store as VS
from voitta_rag_b200.sharded import ShardedIndex

DIM = G.DIM


@pytest.fixture()
def store(monkeypatch):
    monkeypatch.setenv("QDRANT_COLLECTION", "per_query_filters_test")
    monkeypatch.setenv("EMBEDDING_DIMENSION", str(DIM))
    VS._drop_collection("per_query_filters_test")
    s = VS.VectorStoreService(_index_factory=lambda: FakeIndex(DIM))
    yield s
    VS._drop_collection("per_query_filters_test")


def filter_specs(folders, n, seed):
    """n distinct _build_filter keyword sets: folder scopes of every kind, date ranges on both fields."""
    rng = np.random.RandomState(seed)
    specs = []
    while len(specs) < n:
        kw = {}
        kind = rng.randint(4)
        if kind == 0:
            kw["folder_filter"] = folders[rng.randint(len(folders))]
        elif kind == 1:
            kw["include_folders"] = sorted(rng.choice(folders, size=rng.randint(1, len(folders)), replace=False).tolist())
        elif kind == 2:
            kw["exclude_folders"] = sorted(rng.choice(folders, size=rng.randint(1, 4), replace=False).tolist())
            kw["exclude_index_folders"] = ["root%d" % rng.randint(3)] if rng.rand() < 0.5 else None
        if kind == 3 or rng.rand() < 0.5:
            lo = 1420070400 + int(rng.randint(0, 250_000_000))
            kw["date_start"], kw["date_end"] = lo, lo + int(rng.randint(20_000_000, 200_000_000))
            kw["date_field"] = ["created", "modified", None][rng.randint(3)]
        if kw not in specs:
            specs.append(kw)
    return specs


def test_search_batch_with_per_query_filters_equals_single_searches(store):
    corpus, _ = G.build_inputs()
    G.replay(store, G.scenario(corpus, [])[:4], corpus, [], VS.ChunkMetadata, {})     # the four ingest calls
    folders = sorted({m["folder_path"] for m in corpus["metas"]})
    qs = _data.make_queries(seed=5, corpus=corpus, nq=300)
    specs = filter_specs(folders, 40, seed=2)
    B = len(qs)
    filters = []
    for i in range(B):
        if i % 9 == 4:
            filters.append(None)
        else:
            # content repeats across distinct dicts (and the scope_key path caches the folded bits)
            kw = dict(specs[(i * 7) % len(specs)])
            if i % 5 == 0:
                kw["scope_key"] = ("user", (i * 7) % len(specs))
            filters.append(kw)
    Q = [q.astype(float).tolist() for q, _ in qs]
    SP = [sp for _, sp in qs]
    got = store.search_batch(Q, limit=10, sparse_queries=SP, filters=filters)
    assert len(got) == B
    n_nonempty = 0
    for i in range(B):
        kw = filters[i] or {}
        want = store.search(Q[i], limit=10, sparse_query=SP[i], **kw)
        assert [(c.id, c.score) for c in got[i]] == [(c.id, c.score) for c in want], f"query {i} ({kw})"
        n_nonempty += bool(want)
    assert n_nonempty > B // 2


def test_search_batch_filters_argument_errors(store):
    corpus, _ = G.build_inputs()
    G.replay(store, G.scenario(corpus, [])[:1], corpus, [], VS.ChunkMetadata, {})
    Q = [corpus["dense"][r].astype(float).tolist() for r in range(3)]
    with pytest.raises(ValueError, match="one entry per query"):
        store.search_batch(Q, filters=[None, None])
    with pytest.raises(ValueError, match="not both"):
        store.search_batch(Q, folder_filter=corpus["metas"][0]["folder_path"], filters=[None, None, None])
    with pytest.raises(ValueError, match="not both"):
        store.search_batch(Q, date_start=1500000000, filters=[None, None, None])
    # every entry unfiltered: the same as no filter at all
    assert ([[c.id for c in r] for r in store.search_batch(Q, filters=[None, None, None])]
            == [[c.id for c in r] for r in store.search_batch(Q)])


def _worker(rank, world, port, ret):
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        n, dim = 3000, 32
        corpus = _data.make_corpus(seed=21, n=n, dim=dim, vocab=600)
        queries = _data.make_queries(seed=8, corpus=corpus, nq=300)
        coded = _coded.code_corpus(corpus)
        cuts = [0, 1100, n]
        shard = FakeShardIndex(coded, cuts[rank], cuts[rank + 1])
        sh = ShardedIndex(shard, rank, world, device=torch.device("cpu"))
        t, df = shard.directory()
        sh.finalize(t, df, shard.n)
        Q = np.stack([q for q, _ in queries])
        SP = [s for _, s in queries]
        folders = [f for f, _ in coded["scope_list"]]
        rng = np.random.RandomState(12)
        distinct = []
        for k in range(120):
            inc = rng.choice(len(folders), size=rng.randint(1, len(folders)), replace=False)
            lo = 1420070400 + int(rng.randint(0, 200_000_000))
            distinct.append((_coded.scope_bits(coded["scope_list"], include=[folders[j] for j in inc]), 1 + k % 2, lo, engine.TS_MAX))
        B = len(Q)
        flts, fo = [], np.full(B, -1, np.int32)
        for i in range(B):
            if i % 11 == 3:
                continue
            bits, field, lo, hi = distinct[(i * 17) % len(distinct)]
            fo[i] = len(flts)
            flts.append(engine.Filter(bits.copy(), field, lo, hi))      # one object per query, contents repeat
        got = sh.search_batch(Q, SP, flts, fo, limit=8, fusion="rrf")
        whole = oracle_c.CorpusC(coded["dense"], coded["csr"], coded["scope"], coded["created"], coded["modified"])
        want = whole.search_batch(Q, SP, [(f.scope_bits, f.ts_field, f.ts_lo, f.ts_hi) for f in flts], fo, limit=8, fusion=2)
        assert np.array_equal(got.counts, want["counts"])
        for i in range(B):
            c = got.counts[i]
            assert np.array_equal(got.rows[i, :c], want["rows"][i, :c]), i
            np.testing.assert_allclose(got.scores[i, :c], want["scores"][i, :c], rtol=1e-12)
        ret[rank] = "ok"
    finally:
        dist.destroy_process_group()


def test_two_rank_gloo_single_collective_batch_with_per_query_filters():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(2, port, ret), nprocs=2, join=True)
    assert dict(ret) == {0: "ok", 1: "ok"}
