"""Tensor hand-off (SURVEY 8 f-4): dense queries that already live on the GPU (the embedding model's
output, embedding.py:76-86) go through vb_search_dev / vb_stage_dev.  The device path must return
exactly what the host path returns for the same values, and against the oracle like every other path."""
import numpy as np
import pytest

import _data
import _coded
from _parity import assert_same_list, assert_same_ranking
from oracle import oracle_c

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def world():
    from voitta_rag_b200 import engine
    n, dim = 30000, 96
    corpus = _data.make_corpus(seed=21, n=n, dim=dim, vocab=2500)
    queries = _data.make_queries(seed=22, corpus=corpus, nq=24)
    coded = _coded.code_corpus(corpus)
    cc = oracle_c.CorpusC(coded["dense"], coded["csr"], coded["scope"], coded["created"], coded["modified"])
    ix = engine.Index(dim)
    ix.upsert(coded["dense"], coded["csr"], coded["scope"], coded["created"], coded["modified"])
    folders = [f for f, _ in coded["scope_list"]]
    flt = (_coded.scope_bits(coded["scope_list"], include=folders[:8]), 2, 1450000000, _coded.TS_MAX)
    return dict(dim=dim, queries=queries, cc=cc, ix=ix, engine=engine, flt=flt)


@pytest.mark.parametrize("B", [1, 3, 24])
@pytest.mark.parametrize("fusion", ["weighted", "rrf"])
def test_device_queries_equal_host_queries_and_oracle(world, B, fusion):
    import torch
    w = world
    eng, ix = w["engine"], w["ix"]
    Q = np.stack([q for q, _ in w["queries"][:B]]).astype(np.float32)
    SP = [s for _, s in w["queries"][:B]]
    fo = np.zeros(B, np.int32)
    host = ix.search_batch(Q, SP, [eng.Filter(*w["flt"])], fo, limit=10, fusion=fusion, branches=True)
    h2d_host = ix.stats()["last_h2d_bytes"]
    # produced on a side stream, right before the call: the library must order its copy after it
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        half = torch.from_numpy(Q * 0.5).to("cuda:0", non_blocking=False)
        for _ in range(20):                                # keep the stream busy so a missing wait would show
            junk = torch.randn(1 << 20, device="cuda:0").sum()
        qd = half + half                                   # exactly Q again
        dev = ix.search_batch(qd, SP, [eng.Filter(*w["flt"])], fo, limit=10, fusion=fusion, branches=True)
    h2d_dev = ix.stats()["last_h2d_bytes"]
    assert h2d_host - h2d_dev >= B * w["dim"] * 4 - 64, "the query rows must not be uploaded from the host"
    for i in range(B):
        assert dev.hits(i) == host.hits(i)
        assert dev.branch(i, "dense") == host.branch(i, "dense")
        assert dev.branch(i, "sparse") == host.branch(i, "sparse")
    want = w["cc"].search_batch(Q, SP, [w["flt"]], fo, limit=10, fusion={"weighted": 1, "rrf": 2}[fusion])
    for i in range(B):
        ws = [(int(want["sparse_rows"][i, j]), float(want["sparse_scores"][i, j])) for j in range(want["sparse_counts"][i])]
        assert_same_list(dev.branch(i, "sparse"), ws, what=f"device-query sparse q{i}")
        wd = [(int(want["dense_rows"][i, j]), float(want["dense_scores"][i, j])) for j in range(want["dense_counts"][i])]
        assert_same_ranking(dev.branch(i, "dense"), wd, rel_tol=2e-5, abs_tol=2e-5, what=f"device-query dense q{i}")


def test_device_queries_through_the_pipelined_stream(world):
    import torch
    w = world
    eng, ix = w["engine"], w["ix"]
    B = 8
    batches = []
    for r in range(3):
        Q = np.stack([q for q, _ in w["queries"][r * B:(r + 1) * B]]).astype(np.float32)
        SP = [s for _, s in w["queries"][r * B:(r + 1) * B]]
        batches.append((Q, SP))
    fo = np.zeros(B, np.int32)
    host = [ix.search_batch(Q, SP, [eng.Filter(*w["flt"])], fo, limit=10, fusion="rrf") for Q, SP in batches]
    packed = (ix.pack(torch.from_numpy(Q).cuda(), SP, [eng.Filter(*w["flt"])], fo, limit=10, fusion="rrf") for Q, SP in batches)
    got = [[r.hits(i) for i in range(B)] for r in ix.search_stream(packed)]
    assert got == [[h.hits(i) for i in range(B)] for h in host]


def test_non_finite_device_query_is_reported(world):
    import torch
    w = world
    eng, ix = w["engine"], w["ix"]
    Q = np.stack([q for q, _ in w["queries"][:4]]).astype(np.float32)
    qd = torch.from_numpy(Q).cuda()
    qd[2, 5] = float("nan")
    with pytest.raises(eng.B200Error, match="NaN or inf"):
        ix.search_batch(qd, None, limit=5, fusion="dense")
    qd[2, 5] = float("inf")
    with pytest.raises(eng.B200Error, match="NaN or inf"):
        ix.search_batch(qd, None, limit=5, fusion="dense")
    qd[2, 5] = 0.25                                        # and the index keeps working afterwards
    ok = ix.search_batch(qd, None, limit=5, fusion="dense")
    assert len(ok.hits(2)) == 5


def test_wrong_device_pointer_is_refused(world):
    w = world
    eng, ix = w["engine"], w["ix"]

    class FakeTensor:                                     # a "CUDA tensor" whose pointer is host memory
        is_cuda = True

        def __init__(self, a):
            self.a = a
            self.shape = a.shape
            self.dtype = None

        def dim(self):
            return self.a.ndim

        def data_ptr(self):
            return self.a.ctypes.data

    import torch
    a = np.zeros((1, w["dim"]), np.float32)
    t = FakeTensor(a)
    t.dtype = torch.float32
    t.is_contiguous = lambda: True
    t.device = torch.device("cuda:0")
    with pytest.raises(eng.B200Error, match="not a device pointer"):
        ix.search_batch(t, None, limit=5, fusion="dense")


def test_vector_store_service_accepts_cuda_tensors(monkeypatch):
    """The drop-in class: `search(tensor)` and `search_batch(tensor)` return what the list[float] calls return
    (the reference's embed_query ends in .tolist(), embedding.py:76-86; the tensor form skips that hop)."""
    import torch
    from golden import make_golden as G
    from voitta_rag_b200 import vector_store as VS
    name = "gpu_device_queries"
    corpus, queries = G.build_inputs()
    monkeypatch.setenv("QDRANT_COLLECTION", name)
    monkeypatch.setenv("EMBEDDING_DIMENSION", str(corpus["dense"].shape[1]))
    VS._drop_collection(name)
    store = VS.VectorStoreService()
    n = len(corpus["texts"])
    chunks = [(corpus["texts"][r], corpus["dense"][r].astype(float).tolist(), VS.ChunkMetadata(**corpus["metas"][r])) for r in range(n)]
    store.store_chunks(chunks, [corpus["sparse"][r] for r in range(n)])
    folders = sorted({m["folder_path"] for m in corpus["metas"]})
    for qv, sq in queries[:6]:
        for kw in ({}, {"include_folders": folders[:3]}, {"exclude_folders": folders[:1], "date_start": 1500000000, "date_field": "modified"}):
            want = store.search(qv.astype(float).tolist(), limit=7, sparse_query=sq, **kw)
            got = store.search(torch.from_numpy(qv.astype(np.float32)).cuda(), limit=7, sparse_query=sq, **kw)
            assert [(c.id, c.score) for c in got] == [(c.id, c.score) for c in want]
    Q = np.stack([q for q, _ in queries[:6]]).astype(np.float32)
    SQ = [s for _, s in queries[:6]]
    want = store.search_batch(Q, limit=5, sparse_queries=SQ, include_folders=folders[:4])
    got = store.search_batch(torch.from_numpy(Q).cuda(), limit=5, sparse_queries=SQ, include_folders=folders[:4])
    assert [[(c.id, c.score) for c in r] for r in got] == [[(c.id, c.score) for c in r] for r in want]
    with pytest.raises(ValueError, match="dimension"):
        store.search(torch.zeros(3, device="cuda"), limit=3)
    VS._drop_collection(name)
