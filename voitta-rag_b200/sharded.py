"""Row-sharded multi-GPU search: one process per GPU, ``torch.distributed`` for the plumbing.

The corpus is row-partitioned (contiguous blocks; dense rows, postings, filter columns and
tombstones all follow the same row -> shard map).  Queries, filters and the IDF inputs are
replicated.  Each rank computes the exact top-k' of both branches over its shard
(``vb_search_local``); the exchange step of the path is an all-gather of those candidates
(``[2][B][k']`` packed u64 per rank — NCCL over NVLink on GPUs, gloo in the CPU tests); every rank
then merges n_shards*k' -> k' per branch and only THEN fuses (min-max and ranks are global
properties; fusing per shard would be wrong) — ``vb_merge_fuse``.  That all-gather is the one collective
of a batch.

IDF needs global statistics (N = live points, df per term).  They are host-owned: ``finalize()``
all-gathers each shard's (term, df) directory once and keeps the summed table, so the per-query
weights are computed identically on every rank without a per-query collective.
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.distributed as dist


class ShardedIndex:
    def __init__(self, index, rank: int, world: int, group=None, device=None):
        """``index``: this rank's engine.Index (created with row_base = first global row of the shard)."""
        self.index = index
        self.rank, self.world, self.group = rank, world, group
        self.device = device if device is not None else torch.device("cuda", index.device)
        self.terms_g: np.ndarray | None = None
        self.df_g: np.ndarray | None = None
        self.n_live_g = 0
        self._bufs: dict = {}
        self._idf_cache: dict = {}
        # one CUDA stream carries the library's kernels AND the collective, so they are ordered
        # without host synchronisation
        self.stream = None
        if self.device.type == "cuda":
            self.stream = torch.cuda.Stream(self.device)
            self.index.set_option("stream", self.stream.cuda_stream)

    def _stream_ctx(self):
        import contextlib
        return torch.cuda.stream(self.stream) if self.stream is not None else contextlib.nullcontext()

    # ---- global IDF statistics ----------------------------------------------------------------
    def _all_gather_var(self, arr: np.ndarray) -> list[np.ndarray]:
        """all-gather of variable-length int64 arrays (pad to the max length)."""
        if self.world == 1:
            return [arr.astype(np.int64)]
        n = torch.tensor([arr.size], dtype=torch.int64, device=self.device)
        sizes = [torch.zeros_like(n) for _ in range(self.world)]
        dist.all_gather(sizes, n, group=self.group)
        m = max(int(s.item()) for s in sizes)
        buf = torch.zeros(max(m, 1), dtype=torch.int64, device=self.device)
        buf[:arr.size] = torch.from_numpy(arr.astype(np.int64)).to(self.device)
        out = [torch.zeros_like(buf) for _ in range(self.world)]
        dist.all_gather(out, buf, group=self.group)
        return [o[:int(s.item())].cpu().numpy() for o, s in zip(out, sizes)]

    def finalize(self, local_terms: np.ndarray, local_df: np.ndarray, n_live_local: int) -> None:
        """Exchange the shard term directories; afterwards ``idf_weights`` needs no collective."""
        packed = (local_terms.astype(np.int64) << 32) | local_df.astype(np.int64)
        parts = self._all_gather_var(packed)
        allp = np.concatenate(parts) if parts else np.zeros(0, np.int64)
        terms = (allp >> 32).astype(np.uint32)
        df = (allp & 0xFFFFFFFF).astype(np.int64)
        order = np.argsort(terms, kind="stable")
        terms, df = terms[order], df[order]
        uniq, start = np.unique(terms, return_index=True)
        self.terms_g = uniq
        self.df_g = np.add.reduceat(df, start) if len(df) else np.zeros(0, np.int64)
        n = torch.tensor([n_live_local], dtype=torch.int64, device=self.device)
        if self.world > 1:
            dist.all_reduce(n, group=self.group)
        self.n_live_g = int(n.item())
        self._idf_cache = {}

    def finalize_from_queries(self, sparse_batches) -> None:
        """Cheaper variant for static benchmark corpora: only the terms that occur in the given
        query batches are exchanged (df via vb_term_stats on each shard)."""
        terms = sorted({int(t) for sp in sparse_batches for s in sp if s is not None for t in s[0]})
        t = np.asarray(terms, dtype=np.uint32)
        df, n_live = self.index.term_stats(t)
        self.finalize(t, np.asarray(df, dtype=np.int64), n_live)

    def idf_weights(self, sparse):
        """qdrant's IDF modifier with GLOBAL statistics (local_collection.py _rescore_idf).  One flattening pass, one
        factor per DISTINCT term of the batch (cached; math.log as in the single-shard path, so the products are the
        same doubles), one vectorised multiply.  Returns engine.FlatSparse."""
        if sparse is None:
            return None
        from . import engine as _engine
        flat = _engine.flatten_sparse(sparse, len(sparse))
        nnz = int(flat.indptr[-1])
        if nnz == 0:
            return flat
        cache = self._idf_cache          # term -> ln((N - df + 0.5) / (df + 0.5) + 1), emptied by finalize()
        uniq, inv = np.unique(flat.terms[:nnz], return_inverse=True)
        f = np.empty(len(uniq), np.float64)
        for j, t in enumerate(uniq.tolist()):
            v = cache.get(t)
            if v is None:
                v = cache[t] = self._idf_factor(t)
            f[j] = v
        w = np.zeros_like(flat.weights)
        w[:nnz] = flat.weights[:nnz] * f[inv]
        return _engine.FlatSparse(flat.indptr, flat.terms, w)

    def _idf_factor(self, term: int) -> float:
        N, d = self.n_live_g, 0.0
        if len(self.terms_g):
            pos = int(np.searchsorted(self.terms_g, np.uint32(term)))
            if pos < len(self.terms_g) and int(self.terms_g[pos]) == int(term):
                d = float(self.df_g[pos])
        return math.log((N - d + 0.5) / (d + 0.5) + 1.0)

    # ---- query --------------------------------------------------------------------------------
    def _buf(self, name, numel):
        b = self._bufs.get(name)
        if b is None or b.numel() < numel:
            b = torch.zeros(numel, dtype=torch.int64, device=self.device)
            if b.is_cuda:
                torch.cuda.synchronize(self.device)
            self._bufs[name] = b
        return b[:numel]

    def search_batch(self, queries, sparse=None, filters=None, filter_of=None, limit=10, kprime=None,
                     fusion="weighted", sparse_weight=0.1, branches=False):
        """Same call shape and result as engine.Index.search_batch; identical on every rank."""
        q = queries if getattr(queries, "is_cuda", False) else np.ascontiguousarray(queries, dtype=np.float32)
        B = int(q.shape[0])
        any_sparse = sparse is not None and any(s is not None and len(s[0]) for s in sparse)
        if kprime is None:
            kprime = limit * 3 if (any_sparse and fusion != "dense") else limit
        weighted = self.idf_weights(sparse) if any_sparse else None
        staged = self.index.stage(q, weighted, filters, filter_of, limit=limit, kprime=kprime, fusion=fusion,
                                  sparse_weight=sparse_weight, apply_idf=False, branches=branches)
        try:
            for attempt in range(2):
                if attempt:
                    self.index.set_option("safe_mode", 1)     # some shard overflowed: every rank re-runs
                res = self.run_staged(staged, B, kprime)
                if res is not None:
                    return res
        finally:
            self.index.set_option("safe_mode", 0)
        raise RuntimeError("candidate list overflow even in safe mode")

    def pack(self, queries, sparse=None, filters=None, filter_of=None, limit=10, kprime=None,
             fusion="weighted", sparse_weight=0.1, branches=False):
        """Host buffers of one batch with the GLOBAL idf already applied (reusable across calls)."""
        # (a torch CUDA tensor on this rank's device goes through as it is: vb_stage_dev, no H2D copy of the vectors)
        q = queries if getattr(queries, "is_cuda", False) else np.ascontiguousarray(queries, dtype=np.float32)
        any_sparse = sparse is not None and any(s is not None and len(s[0]) for s in sparse)
        if kprime is None:
            kprime = limit * 3 if (any_sparse and fusion != "dense") else limit
        weighted = self.idf_weights(sparse) if any_sparse else None
        p = self.index.pack(q, weighted, filters, filter_of, limit=limit, kprime=kprime, fusion=fusion,
                            sparse_weight=sparse_weight, apply_idf=False, branches=branches)
        p.kprime = kprime
        return p

    def search_packed(self, packed):
        """stage (H2D) -> local branches -> all-gather -> merge + fuse -> fetch (D2H) on prepared buffers."""
        try:
            for attempt in range(2):
                if attempt:
                    self.index.set_option("safe_mode", 1)
                staged = self.index.stage_packed(packed)
                res = self.run_staged(staged, packed.B, packed.kprime)
                if res is not None:
                    return res
        finally:
            self.index.set_option("safe_mode", 0)
        raise RuntimeError("candidate list overflow even in safe mode")

    def search_stream(self, packed_iter):
        """Pipelined ``search_packed`` over a stream of prepared batches (two in flight per rank):
        staging + H2D of batch i+1 overlap the kernels / all-gather of batch i.  Yields in order."""
        prev = None
        slot = 0
        import time
        t = self.host_ms = {"stage": 0.0, "enqueue": 0.0, "fetch": 0.0, "batches": 0}   # host wall time per call site (diagnostic)
        try:
            for packed in packed_iter:
                self.index.set_option("slot", slot)
                t0 = time.perf_counter()
                staged = self.index.stage_packed(packed)
                t1 = time.perf_counter()
                self._enqueue(packed.B, packed.kprime)
                t2 = time.perf_counter()
                t["stage"] += 1e3 * (t1 - t0); t["enqueue"] += 1e3 * (t2 - t1); t["batches"] += 1
                if prev is not None:
                    self.index.set_option("slot", slot ^ 1)
                    res = self.index.fetch(prev, allow_overflow=True)
                    t["fetch"] += 1e3 * (time.perf_counter() - t2)
                    if res is None:
                        raise RuntimeError("candidate overflow in a pipelined search; use search_packed")
                    yield res
                prev = staged
                slot ^= 1
            if prev is not None:
                self.index.set_option("slot", slot ^ 1)
                res = self.index.fetch(prev, allow_overflow=True)
                if res is None:
                    raise RuntimeError("candidate overflow in a pipelined search; use search_packed")
                yield res
        finally:
            self.index.set_option("slot", 0)

    def _enqueue(self, B: int, kprime: int):
        """local branches -> all-gather -> merge + fuse, all asynchronous on this rank's stream."""
        words = self.index.cand_block_words(B, kprime)
        local = self._buf("local", words)
        gathered = self._buf("gathered", words * self.world)
        with self._stream_ctx():
            self.index.run_local(local.data_ptr())
            if self.world > 1:
                dist.all_gather_into_tensor(gathered, local, group=self.group)
            else:
                gathered.copy_(local)
            self.index.run_fuse(self.world, gathered.data_ptr())

    def run_staged(self, staged, B: int, kprime: int):
        """Device part of one sharded search on an already staged batch: local branches ->
        all-gather of the candidate blocks (the path's ONE exchange step) -> merge -> fuse -> fetch."""
        self._enqueue(B, kprime)
        return self.index.fetch(staged, allow_overflow=True)
