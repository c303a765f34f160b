"""world_size-2 test of the row-sharded host logic (voitta_rag_b200.sharded) on CPU with the gloo
backend: global IDF exchange, candidate all-gather, merge-then-fuse.  The per-shard engine is a
test double backed by the C oracle; the GPU version of the same flow is
tests/test_gpu_engine.py::test_two_shards_merged_and_staged_equal_single_index."""
import ctypes
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import _data
import _coded
from oracle import oracle as O
from oracle import oracle_c
from voitta_rag_b200 import engine
from voitta_rag_b200.sharded import ShardedIndex


class FakeShardIndex:
    device = -1

    def __init__(self, coded, lo, hi):
        ip, tm, vl = coded["csr"]
        self.row_base = lo
        self.csr = (ip[lo:hi + 1] - ip[lo], tm[ip[lo]:ip[hi]], vl[ip[lo]:ip[hi]])
        self.cc = oracle_c.CorpusC(coded["dense"][lo:hi], self.csr, coded["scope"][lo:hi], coded["created"][lo:hi],
                                   coded["modified"][lo:hi])
        self.n = hi - lo

    def directory(self):
        t, c = np.unique(self.csr[1], return_counts=True)
        return t.astype(np.uint32), c.astype(np.int64)

    @staticmethod
    def cand_block_words(B, k):
        return 2 * B * k + 1

    def set_option(self, key, value):
        pass

    def stage(self, queries, sparse=None, filters=None, filter_of=None, limit=10, kprime=None, fusion="weighted",
              sparse_weight=0.1, apply_idf=True, branches=False, need_corpus=True):
        assert not apply_idf
        self.st = dict(q=queries, sp=sparse, fl=filters, fo=filter_of, limit=limit, k=kprime, fusion=fusion, w=sparse_weight)
        return "staged"

    def run_local(self, ptr):
        st = self.st
        fl = None if not st["fl"] else [(f.scope_bits, f.ts_field, f.ts_lo, f.ts_hi) for f in st["fl"]]
        out = self.cc.search_batch(st["q"], st["sp"], fl, st["fo"], st["limit"], st["k"], 1 if st["sp"] is not None else 0,
                                   st["w"], apply_idf=False)
        B, k = len(st["q"]), st["k"]
        keys = np.zeros(2 * B * k + 1, np.uint64)
        kv = keys[:-1].reshape(2, B, k)
        for br, name in enumerate(("dense", "sparse")):
            for i in range(B):
                c = int(out[f"{name}_counts"][i])
                kv[br, i, :c] = engine.pack_keys(out[f"{name}_scores"][i, :c], out[f"{name}_rows"][i, :c] + self.row_base)
        ctypes.memmove(ptr, keys.ctypes.data, keys.nbytes)

    def run_fuse(self, n_shards, ptr):
        st = self.st
        B, k, limit = len(st["q"]), st["k"], st["limit"]
        words = 2 * B * k + 1
        g = np.ctypeslib.as_array((ctypes.c_uint64 * (n_shards * words)).from_address(ptr)).reshape(n_shards, words)
        assert not g[:, -1].any()
        g = g[:, :-1].reshape(n_shards, 2, B, k)
        res = engine.SearchResult(np.zeros((B, limit), np.uint64), np.zeros((B, limit)), np.zeros(B, np.int32))
        for i in range(B):
            lists = []
            for br in range(2):
                kk = np.sort(g[:, br, i, :].ravel())[::-1]
                kk = kk[kk != 0][:k]
                sc, rows = engine.unpack_keys(kk)
                lists.append([O.ScoredPoint(str(int(r)), float(s), {}, int(r)) for s, r in zip(sc, rows)])
            sp = st["sp"]
            has_sparse = sp is not None and sp[i] is not None and len(sp[i][0])
            if not has_sparse:
                fused = [(p.id, p.score, p) for p in lists[0][:limit]]
            elif st["fusion"] == "rrf":
                fused = O.reciprocal_rank_fusion(lists, limit)
            else:
                fused = O.weighted_fusion(lists[0], lists[1], limit, st["w"])
            res.counts[i] = len(fused)
            for j, (pid, s_, _) in enumerate(fused):
                res.rows[i, j], res.scores[i, j] = int(pid), s_
        self.res = res

    def fetch(self, staged, allow_overflow=False):
        return self.res


def _worker(rank, world, port, ret):
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        n, dim = 3000, 32
        corpus = _data.make_corpus(seed=21, n=n, dim=dim, vocab=600)
        queries = _data.make_queries(seed=4, corpus=corpus, nq=6)
        coded = _coded.code_corpus(corpus)
        cuts = [0, 1100, n]
        shard = FakeShardIndex(coded, cuts[rank], cuts[rank + 1])
        sh = ShardedIndex(shard, rank, world, device=torch.device("cpu"))
        t, df = shard.directory()
        sh.finalize(t, df, shard.n)
        assert sh.n_live_g == n
        Q = np.stack([q for q, _ in queries])
        SP = [s for _, s in queries]
        SP[2] = None                                            # a dense-only query inside the batch
        bits = _coded.scope_bits(coded["scope_list"], include=[f for f, _ in coded["scope_list"]][:7])
        flt = engine.Filter(bits, 2, 1450000000, engine.TS_MAX)
        whole = oracle_c.CorpusC(coded["dense"], coded["csr"], coded["scope"], coded["created"], coded["modified"])
        for fusion in ("weighted", "rrf"):
            got = sh.search_batch(Q, SP, [flt], np.zeros(len(Q), np.int32), limit=8, fusion=fusion, sparse_weight=0.25)
            want = whole.search_batch(Q, SP, [(bits, 2, 1450000000, engine.TS_MAX)], np.zeros(len(Q), np.int32), limit=8,
                                      fusion={"weighted": 1, "rrf": 2}[fusion], sparse_weight=0.25)
            assert np.array_equal(got.counts, want["counts"]), (fusion, got.counts, want["counts"])
            for i in range(len(Q)):
                c = got.counts[i]
                assert np.array_equal(got.rows[i, :c], want["rows"][i, :c]), (fusion, i)
                np.testing.assert_allclose(got.scores[i, :c], want["scores"][i, :c], rtol=1e-12)
        ret[rank] = "ok"
    finally:
        dist.destroy_process_group()


def test_two_rank_gloo_single_collective_search():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(2, port, ret), nprocs=2, join=True)
    assert dict(ret) == {0: "ok", 1: "ok"}
