"""ctypes binding of libvoitta_b200.so (include/voitta_b200.h) and the ``Index`` handle.

This is the thin layer the north_star asks for: Python host code calls CUDA through the C ABI;
numpy arrays (host) or raw device pointers (torch tensors' ``data_ptr()``) cross the boundary.
There is no CPU fallback: if the library is missing or no sm_100 device is present, every
compute call raises ``B200Error``.
"""
from __future__ import annotations

import ctypes as C
import itertools
from dataclasses import dataclass
from pathlib import Path

import numpy as np

import os

HERE = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ["VB200_LIB"]) if os.environ.get("VB200_LIB") else HERE / "libvoitta_b200.so"   # (debug build: bounds checks)

TS_MISSING = -(2 ** 63)
TS_MIN = -(2 ** 63) + 1
TS_MAX = 2 ** 63 - 1
FUSE_DENSE_ONLY, FUSE_WEIGHTED, FUSE_RRF = 0, 1, 2
FUSION = {"dense": FUSE_DENSE_ONLY, "weighted": FUSE_WEIGHTED, "rrf": FUSE_RRF}
TS_NONE, TS_CREATED, TS_MODIFIED = 0, 1, 2
MAX_KPRIME = 1024


class B200Error(RuntimeError):
    pass


# pointer fields are declared c_void_p (same ABI): an integer address is assigned directly, which costs a fifth of
# ndarray.ctypes.data_as(POINTER(...)) — the B = 1 call path builds two of these structs per search
class _Filter(C.Structure):
    _fields_ = [("scope_bits", C.c_void_p), ("scope_words", C.c_uint32),
                ("ts_field", C.c_int32), ("ts_lo", C.c_int64), ("ts_hi", C.c_int64)]


class _QueryBatch(C.Structure):
    _fields_ = [("n_queries", C.c_uint32), ("dense", C.c_void_p),
                ("sp_indptr", C.c_void_p), ("sp_term", C.c_void_p),
                ("sp_weight", C.c_void_p), ("apply_idf", C.c_int32),
                ("n_filters", C.c_uint32), ("filters", C.c_void_p),
                ("filter_of", C.c_void_p), ("limit", C.c_uint32), ("kprime", C.c_uint32),
                ("fusion", C.c_int32), ("sparse_weight", C.c_double)]


class _Result(C.Structure):
    _fields_ = [("rows", C.c_void_p), ("scores", C.c_void_p),
                ("counts", C.c_void_p),
                ("dense_rows", C.c_void_p), ("dense_scores", C.c_void_p),
                ("dense_counts", C.c_void_p),
                ("sparse_rows", C.c_void_p), ("sparse_scores", C.c_void_p),
                ("sparse_counts", C.c_void_p)]


class _Stats(C.Structure):
    _fields_ = [("n_rows", C.c_uint64), ("n_live", C.c_uint64), ("nnz", C.c_uint64), ("n_terms", C.c_uint64),
                ("searches", C.c_uint64), ("queries", C.c_uint64), ("overflow_reruns", C.c_uint64),
                ("last_search_ms", C.c_double), ("last_dense_ms", C.c_double), ("last_sparse_ms", C.c_double),
                ("last_select_ms", C.c_double), ("last_mask_ms", C.c_double), ("last_fuse_ms", C.c_double),
                ("last_dense_path", C.c_uint32), ("last_launches", C.c_uint32), ("device_bytes", C.c_uint64),
                ("last_h2d_bytes", C.c_uint64), ("last_d2h_bytes", C.c_uint64), ("last_dense_passes", C.c_uint64),
                ("last_big_rows", C.c_uint64), ("last_dense_big_ms", C.c_double), ("last_sparse_big_ms", C.c_double),
                ("dim", C.c_uint64), ("row_base", C.c_uint64), ("index_builds", C.c_uint64), ("delta_rows", C.c_uint64),
                ("last_overflow_lists", C.c_uint32), ("last_overflow_first", C.c_uint32),
                ("last_sel_rows", C.c_uint32), ("last_sel_used", C.c_uint32)]


# every symbol include/voitta_b200.h declares
ABI_VERSION = 4          # include/voitta_b200.h VB_ABI_VERSION

EXPORTS = ["vb_abi_version", "vb_last_error", "vb_create", "vb_destroy", "vb_upsert", "vb_upsert_dev",
           "vb_delete_rows", "vb_optimize", "vb_term_stats", "vb_search", "vb_search_local", "vb_merge_fuse",
           "vb_stage", "vb_run_local", "vb_run_fuse", "vb_fetch", "vb_stage_dev", "vb_search_dev",
           "vb_set_option", "vb_get_stats", "vb_get_timeline", "vb_sync", "vb_save", "vb_load"]

_lib = None


def load_library():
    """dlopen the in-tree library.  Never builds and never falls back."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise B200Error(f"{LIB_PATH} not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(there is no CPU fallback)")
    lib = C.CDLL(str(LIB_PATH))
    vp, u64p, u32p = C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)
    lib.vb_abi_version.restype = C.c_int
    if lib.vb_abi_version() != ABI_VERSION:
        raise B200Error(f"{LIB_PATH} has ABI version {lib.vb_abi_version()}, this module binds version {ABI_VERSION}: rebuild it")
    lib.vb_last_error.restype = C.c_char_p
    lib.vb_create.argtypes = [C.c_int32, C.c_int32, C.c_uint64, C.c_uint64, C.POINTER(vp)]
    lib.vb_destroy.argtypes = [vp]
    lib.vb_destroy.restype = None
    lib.vb_upsert.argtypes = [vp, C.c_uint64, vp, vp, vp, vp, vp, vp, vp, u64p]
    lib.vb_upsert_dev.argtypes = [vp, C.c_uint64, vp, vp, vp, vp, vp, vp, vp, u64p]
    lib.vb_delete_rows.argtypes = [vp, C.c_uint64, vp]
    lib.vb_optimize.argtypes = [vp]
    lib.vb_term_stats.argtypes = [vp, C.c_uint32, vp, vp, u64p]
    lib.vb_search.argtypes = [vp, C.POINTER(_QueryBatch), C.POINTER(_Result)]
    lib.vb_search_local.argtypes = [vp, C.POINTER(_QueryBatch), vp]
    lib.vb_merge_fuse.argtypes = [vp, C.POINTER(_QueryBatch), C.c_uint32, vp, C.POINTER(_Result)]
    lib.vb_stage.argtypes = [vp, C.POINTER(_QueryBatch), C.c_int32, C.c_int32]
    lib.vb_stage_dev.argtypes = [vp, C.POINTER(_QueryBatch), vp, vp, C.c_int32, C.c_int32]
    lib.vb_search_dev.argtypes = [vp, C.POINTER(_QueryBatch), vp, vp, C.POINTER(_Result)]
    lib.vb_run_local.argtypes = [vp, vp]
    lib.vb_run_fuse.argtypes = [vp, C.c_uint32, vp]
    lib.vb_fetch.argtypes = [vp, C.POINTER(_Result), C.POINTER(C.c_int32)]
    lib.vb_set_option.argtypes = [vp, C.c_char_p, C.c_int64]
    lib.vb_get_stats.argtypes = [vp, C.POINTER(_Stats)]
    lib.vb_sync.argtypes = [vp]
    lib.vb_get_timeline.argtypes = [vp, vp, C.c_uint32, C.POINTER(C.c_uint32)]
    lib.vb_save.argtypes = [vp, C.c_char_p]
    lib.vb_load.argtypes = [C.c_char_p, C.c_int32, C.POINTER(vp)]
    _lib = lib
    return lib


def _ptr(a, ctype=None):
    """Address of a numpy array's buffer (or None) for a c_void_p struct field; the caller keeps the array alive."""
    return a.ctypes.data if a is not None else None


def _vp(a):
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    return C.c_void_p(a.ctypes.data)


@dataclass
class Filter:
    """One evaluated filter (see vb_filter).  ``scope_bits``: uint32 words over scope ids or None."""
    scope_bits: np.ndarray | None = None
    ts_field: int = TS_NONE
    ts_lo: int = TS_MIN
    ts_hi: int = TS_MAX


@dataclass
class SearchResult:
    rows: np.ndarray            # [B, limit] uint64
    scores: np.ndarray          # [B, limit] float64
    counts: np.ndarray          # [B] int32
    dense_rows: np.ndarray | None = None
    dense_scores: np.ndarray | None = None
    dense_counts: np.ndarray | None = None
    sparse_rows: np.ndarray | None = None
    sparse_scores: np.ndarray | None = None
    sparse_counts: np.ndarray | None = None

    def hits(self, q: int):
        c = int(self.counts[q])
        return list(zip(self.rows[q, :c].tolist(), self.scores[q, :c].tolist()))

    def branch(self, q: int, which: str):
        rows, sc, cn = ((self.dense_rows, self.dense_scores, self.dense_counts) if which == "dense"
                        else (self.sparse_rows, self.sparse_scores, self.sparse_counts))
        c = int(cn[q])
        return [(int(rows[q, i]), float(sc[q, i])) for i in range(c)]


def pack_keys(scores, rows) -> np.ndarray:
    """Candidate keys as the kernels build them (csrc/common.cuh): hi = monotone map of the fp32
    score, lo = ~row, so that a larger key means (higher score, then lower row).  0 = empty."""
    s = np.asarray(scores, dtype=np.float32) + np.float32(0.0)
    u = s.view(np.uint32).astype(np.uint64)
    o = np.where(u & 0x80000000, (~u) & 0xFFFFFFFF, u ^ 0x80000000)
    r = (~np.asarray(rows, dtype=np.uint32)).astype(np.uint64)
    return ((o << np.uint64(32)) | r).astype(np.uint64)


def unpack_keys(keys):
    """Inverse of pack_keys -> (scores float32, rows uint32)."""
    k = np.asarray(keys, dtype=np.uint64)
    o = (k >> np.uint64(32)).astype(np.uint64)
    u = np.where(o & 0x80000000, o ^ 0x80000000, (~o) & 0xFFFFFFFF).astype(np.uint32)
    return u.view(np.float32), (~(k & np.uint64(0xFFFFFFFF)).astype(np.uint32))


class FlatSparse:
    """A batch of sparse queries in flattened (CSR) form: indptr int64 [B + 1], terms uint32 [nnz], weights float64
    [nnz].  ``flatten_sparse`` builds it from the reference's per-query ``(indices, values)`` pairs in one pass; the
    sharded layer multiplies the weights by the global IDF in place of a per-term Python loop."""
    __slots__ = ("indptr", "terms", "weights")

    def __init__(self, indptr, terms, weights):
        self.indptr, self.terms, self.weights = indptr, terms, weights

    def __len__(self):
        return len(self.indptr) - 1

    def __getitem__(self, i):
        """Query i as the (indices, values) pair it was built from (sequence protocol: the flat form can stand in for
        the list of pairs anywhere one is read)."""
        if not -len(self) <= i < len(self):
            raise IndexError(i)
        i %= len(self)
        lo, hi = int(self.indptr[i]), int(self.indptr[i + 1])
        return self.terms[lo:hi], self.weights[lo:hi]

    def __iter__(self):
        return (self[i] for i in range(len(self)))


def flatten_sparse(sparse, B: int) -> FlatSparse:
    """[(indices, values) | None] * B -> FlatSparse (one flattening pass for the whole batch: a per-query numpy round trip
    costs ~15 us, 15 ms at B = 1024)."""
    if isinstance(sparse, FlatSparse):
        if len(sparse) != B:
            raise ValueError("one sparse query (or None) per dense query expected")
        return sparse
    if len(sparse) != B:
        raise ValueError("one sparse query (or None) per dense query expected")
    if B == 1:                                               # the reference's own call shape (mcp_server.py:474): no batch machinery
        s0 = sparse[0]
        n0 = 0 if s0 is None else len(s0[0])
        if n0 != (0 if s0 is None else len(s0[1])):
            raise ValueError("sparse indices/values length mismatch")
        indptr = np.array([0, n0], dtype=np.int64)
        if n0 == 0:
            return FlatSparse(indptr, np.zeros(1, np.uint32), np.zeros(1, np.float64))
        idx = np.asarray(s0[0], dtype=np.int64)
        if idx.min() < 0 or idx.max() > 0xFFFFFFFF:
            raise ValueError("sparse index out of uint32 range")
        return FlatSparse(indptr, idx.astype(np.uint32), np.asarray(s0[1], dtype=np.float64))
    lens = np.fromiter((0 if s is None else len(s[0]) for s in sparse), np.int64, B)
    lens_v = np.fromiter((0 if s is None else len(s[1]) for s in sparse), np.int64, B)
    if (lens != lens_v).any():
        raise ValueError("sparse indices/values length mismatch")
    indptr = np.zeros(B + 1, dtype=np.int64)
    np.cumsum(lens, out=indptr[1:])
    nnz = int(indptr[-1])
    terms = np.zeros(max(nnz, 1), dtype=np.uint32)
    weights = np.zeros(max(nnz, 1), dtype=np.float64)
    if nnz:
        parts = [s for s in sparse if s is not None and len(s[0])]
        if all(isinstance(s[0], np.ndarray) and isinstance(s[1], np.ndarray) for s in parts):
            idx = np.concatenate([s[0] for s in parts]).astype(np.int64, copy=False)
            val = np.concatenate([s[1] for s in parts]).astype(np.float64, copy=False)
        else:
            idx = np.fromiter(itertools.chain.from_iterable(s[0] for s in parts), np.int64, nnz)
            val = np.fromiter(itertools.chain.from_iterable(s[1] for s in parts), np.float64, nnz)
        if (idx < 0).any() or (idx > 0xFFFFFFFF).any():
            raise ValueError("sparse index out of uint32 range")
        terms[:nnz] = idx.astype(np.uint32)
        weights[:nnz] = val
    return FlatSparse(indptr, terms, weights)


class _Packed:
    """Keeps the numpy arrays behind a vb_query_batch alive."""

    def __init__(self, dim, queries, sparse, filters, filter_of, limit, kprime, fusion, sparse_weight, apply_idf):
        self.q_dev = None
        self.q_stream = None
        if getattr(queries, "is_cuda", False) and hasattr(queries, "data_ptr"):
            # tensor hand-off (SURVEY 8 f-4): the rows stay on the GPU; NaN / inf are found by the query-prep kernel
            import torch
            t = queries if queries.dim() == 2 else queries[None, :]
            if t.dtype != torch.float32 or not t.is_contiguous():
                t = t.to(torch.float32).contiguous()
            if t.dim() != 2 or t.shape[1] != dim:
                raise ValueError(f"queries must have shape [B, {dim}], got {tuple(t.shape)}")
            self.q_dev = t
            self.q_stream = torch.cuda.current_stream(t.device).cuda_stream
            q = None
            B = int(t.shape[0])
        else:
            q = np.ascontiguousarray(queries, dtype=np.float32)
            if q.ndim == 1:
                q = q[None, :]
            if q.ndim != 2 or q.shape[1] != dim:
                raise ValueError(f"queries must have shape [B, {dim}], got {q.shape}")
            if not np.isfinite(q).all():
                raise ValueError("Query vector must not contain NaN or inf")
            B = q.shape[0]
        self.q = q
        self.B = B
        self.indptr = self.terms = self.weights = None
        if sparse is not None:
            flat = flatten_sparse(sparse, B)
            self.indptr = np.ascontiguousarray(flat.indptr, dtype=np.int64)
            self.terms = np.ascontiguousarray(flat.terms, dtype=np.uint32)
            self.weights = np.ascontiguousarray(flat.weights, dtype=np.float64)
        self.filters = list(filters or [])
        self.bits = [None if f.scope_bits is None else np.ascontiguousarray(f.scope_bits, dtype=np.uint32)
                     for f in self.filters]
        self.cfilters = (_Filter * max(1, len(self.filters)))()
        for i, f in enumerate(self.filters):
            b = self.bits[i]
            self.cfilters[i] = _Filter(_ptr(b, C.c_uint32), 0 if b is None else b.size,
                                       int(f.ts_field), int(f.ts_lo), int(f.ts_hi))
        self.filter_of = None
        if filter_of is not None:
            self.filter_of = np.ascontiguousarray(filter_of, dtype=np.int32)
            if self.filter_of.shape != (B,):
                raise ValueError("filter_of must have one entry per query")
        self.c = _QueryBatch(B, _ptr(self.q, C.c_float), _ptr(self.indptr, C.c_int64), _ptr(self.terms, C.c_uint32),
                             _ptr(self.weights, C.c_double), int(apply_idf), len(self.filters),
                             C.addressof(self.cfilters), _ptr(self.filter_of, C.c_int32),
                             int(limit), int(kprime), int(fusion), float(sparse_weight))


class Index:
    """One shard of the corpus on one GPU (bf16 rows + inverse norms, inverted sparse index,
    filter columns, tombstones)."""

    def __init__(self, dim: int, device: int = 0, row_base: int = 0, capacity_hint: int = 0):
        self._lib = load_library()
        self._h = C.c_void_p()
        self.dim = int(dim)
        self.device = int(device)
        self.row_base = int(row_base)
        self._check(self._lib.vb_create(self.dim, self.device, int(capacity_hint), self.row_base, C.byref(self._h)))

    def _check(self, rc):
        if rc != 0:
            raise B200Error(self._lib.vb_last_error().decode("utf-8", "replace"))

    # ---- snapshot ---------------------------------------------------------------------------
    def save(self, path) -> None:
        """Write the shard's device data (rows, columns, tombstones, forward sparse CSR) to ``path``."""
        self._check(self._lib.vb_save(self._h, str(path).encode()))

    @classmethod
    def load(cls, path, device: int = 0) -> "Index":
        """A new Index on ``device`` from a snapshot written by ``save``."""
        self = cls.__new__(cls)
        self._lib = load_library()
        self._h = C.c_void_p()
        self.device = int(device)
        rc = self._lib.vb_load(str(path).encode(), self.device, C.byref(self._h))
        if rc != 0:
            raise B200Error(self._lib.vb_last_error().decode("utf-8", "replace"))
        st = self.stats()
        self.dim = int(st["dim"])
        self.row_base = int(st["row_base"])
        return self

    def close(self):
        if self._h:
            self._lib.vb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- ingest -----------------------------------------------------------------------------
    def upsert(self, dense, sparse_csr=None, scope_id=None, created=None, modified=None) -> int:
        """Append rows (host arrays).  sparse_csr = (indptr int64 [n+1], terms uint32, values float32)
        with strictly ascending terms inside each row.  Returns the first row id."""
        d = np.ascontiguousarray(dense, dtype=np.float32)
        if d.ndim != 2 or d.shape[1] != self.dim:
            raise ValueError(f"dense must have shape [n, {self.dim}], got {d.shape}")
        n = d.shape[0]
        ip = tm = vl = None
        if sparse_csr is not None:
            ip = np.ascontiguousarray(sparse_csr[0], dtype=np.int64)
            tm = np.ascontiguousarray(sparse_csr[1], dtype=np.uint32)
            vl = np.ascontiguousarray(sparse_csr[2], dtype=np.float32)
            if ip.shape != (n + 1,):
                raise ValueError("sparse indptr must have n+1 entries")
            if tm.size == 0:
                tm = np.zeros(1, np.uint32)
                vl = np.zeros(1, np.float32)
        sc = None if scope_id is None else np.ascontiguousarray(scope_id, dtype=np.uint32)
        cr = None if created is None else np.ascontiguousarray(created, dtype=np.int64)
        mo = None if modified is None else np.ascontiguousarray(modified, dtype=np.int64)
        first = C.c_uint64()
        self._check(self._lib.vb_upsert(self._h, n, _vp(d), _vp(ip), _vp(tm), _vp(vl), _vp(sc), _vp(cr), _vp(mo),
                                        C.byref(first)))
        return int(first.value)

    def upsert_dev(self, n: int, rows_bf16_ptr: int, indptr_ptr=None, terms_ptr=None, vals_ptr=None,
                   scope_ptr=None, created_ptr=None, modified_ptr=None) -> int:
        """Bulk append from device pointers (e.g. torch tensors' data_ptr())."""
        first = C.c_uint64()
        self._check(self._lib.vb_upsert_dev(self._h, int(n), _vp(rows_bf16_ptr), _vp(indptr_ptr), _vp(terms_ptr),
                                            _vp(vals_ptr), _vp(scope_ptr), _vp(created_ptr), _vp(modified_ptr),
                                            C.byref(first)))
        return int(first.value)

    def delete_rows(self, rows) -> None:
        r = np.ascontiguousarray(rows, dtype=np.uint64)
        self._check(self._lib.vb_delete_rows(self._h, r.size, _vp(r)))

    def optimize(self) -> None:
        """Merge the rows appended since the last index build into the inverted index now."""
        self._check(self._lib.vb_optimize(self._h))

    def term_stats(self, terms):
        t = np.ascontiguousarray(terms, dtype=np.uint32)
        df = np.zeros(max(1, t.size), dtype=np.uint64)
        n_live = C.c_uint64()
        self._check(self._lib.vb_term_stats(self._h, t.size, _vp(t if t.size else np.zeros(1, np.uint32)), _vp(df),
                                            C.byref(n_live)))
        return df[:t.size], int(n_live.value)

    # ---- query ------------------------------------------------------------------------------
    def _alloc_result(self, B, limit, kprime, branches):
        r = SearchResult(np.zeros((B, limit), np.uint64), np.zeros((B, limit), np.float64), np.zeros(B, np.int32))
        if branches:
            r.dense_rows = np.zeros((B, kprime), np.uint64)
            r.dense_scores = np.zeros((B, kprime), np.float32)
            r.dense_counts = np.zeros(B, np.int32)
            r.sparse_rows = np.zeros((B, kprime), np.uint64)
            r.sparse_scores = np.zeros((B, kprime), np.float32)
            r.sparse_counts = np.zeros(B, np.int32)
        c = _Result(_ptr(r.rows, C.c_uint64), _ptr(r.scores, C.c_double), _ptr(r.counts, C.c_int32),
                    _ptr(r.dense_rows, C.c_uint64), _ptr(r.dense_scores, C.c_float), _ptr(r.dense_counts, C.c_int32),
                    _ptr(r.sparse_rows, C.c_uint64), _ptr(r.sparse_scores, C.c_float), _ptr(r.sparse_counts, C.c_int32))
        return r, c

    def search_batch(self, queries, sparse=None, filters=None, filter_of=None, limit: int = 10,
                     kprime: int | None = None, fusion: str | int = "weighted", sparse_weight: float = 0.1,
                     apply_idf: bool = True, branches: bool = False) -> SearchResult:
        """Hybrid filtered top-k for a batch (host buffers in/out; one vb_search call)."""
        fz = FUSION[fusion] if isinstance(fusion, str) else int(fusion)
        if kprime is None:
            kprime = limit * 3 if (sparse is not None and fz != FUSE_DENSE_ONLY) else limit
        p = _Packed(self.dim, queries, sparse, filters, filter_of, limit, kprime, fz, sparse_weight, apply_idf)
        res, cres = self._alloc_result(p.B, limit, kprime, branches)
        self._search(p, cres)
        return res

    def _search(self, p, cres):
        if p.q_dev is not None:
            self._check(self._lib.vb_search_dev(self._h, C.byref(p.c), p.q_dev.data_ptr(), p.q_stream, C.byref(cres)))
        else:
            self._check(self._lib.vb_search(self._h, C.byref(p.c), C.byref(cres)))

    @staticmethod
    def cand_block_words(n_queries: int, kprime: int) -> int:
        """u64 words of one shard's candidate block (VB_CAND_BLOCK_WORDS)."""
        return 2 * n_queries * kprime + 1

    def pack(self, queries, sparse=None, filters=None, filter_of=None, limit: int = 10, kprime: int | None = None,
             fusion: str | int = "weighted", sparse_weight: float = 0.1, apply_idf: bool = True, branches: bool = False):
        """Build the host buffers of a vb_query_batch once (numpy arrays + the C struct); pass the
        result to ``search_packed`` any number of times."""
        fz = FUSION[fusion] if isinstance(fusion, str) else int(fusion)
        if kprime is None:
            kprime = limit * 3 if (sparse is not None and fz != FUSE_DENSE_ONLY) else limit
        p = _Packed(self.dim, queries, sparse, filters, filter_of, limit, kprime, fz, sparse_weight, apply_idf)
        p.result = self._alloc_result(p.B, limit, kprime, branches)
        return p

    def search_packed(self, packed) -> SearchResult:
        """vb_search on prepared host buffers: staging, H2D, kernels, D2H and decode, nothing else."""
        res, cres = packed.result
        self._search(packed, cres)
        return res

    def search_stream(self, packed_iter):
        """Pipelined vb_stage/run/fetch over a stream of prepared batches (two in flight): the host
        work and H2D copy of batch i+1 overlap the kernels of batch i.  Yields results in order.
        Every batch still pays its own H2D and D2H copy."""
        prev = None
        slot = 0
        try:
            for packed in packed_iter:
                self.set_option("slot", slot)
                staged = self.stage_packed(packed)
                self.run_local(None)
                self.run_fuse(0, None)
                if prev is not None:
                    self.set_option("slot", slot ^ 1)
                    res = self.fetch(prev, allow_overflow=True)
                    if res is None:
                        raise B200Error("candidate overflow in a pipelined search; use search_packed for this batch")
                    yield res
                prev = staged
                slot ^= 1
            if prev is not None:
                self.set_option("slot", slot ^ 1)
                res = self.fetch(prev, allow_overflow=True)
                if res is None:
                    raise B200Error("candidate overflow in a pipelined search; use search_packed for this batch")
                yield res
        finally:
            self.set_option("slot", 0)

    def search_local(self, cand_dev_ptr: int, queries, sparse=None, filters=None, filter_of=None, limit: int = 10,
                     kprime: int | None = None, fusion: str | int = "weighted", sparse_weight: float = 0.1):
        """Shard-local branch top-k' left on the device (all-gather payload); weights carry global IDF."""
        fz = FUSION[fusion] if isinstance(fusion, str) else int(fusion)
        if kprime is None:
            kprime = limit * 3
        p = _Packed(self.dim, queries, sparse, filters, filter_of, limit, kprime, fz, sparse_weight, False)
        self._check(self._lib.vb_search_local(self._h, C.byref(p.c), _vp(cand_dev_ptr)))

    def merge_fuse(self, gathered_dev_ptr: int, n_shards: int, queries, sparse=None, limit: int = 10,
                   kprime: int | None = None, fusion: str | int = "weighted", sparse_weight: float = 0.1,
                   branches: bool = False) -> SearchResult:
        fz = FUSION[fusion] if isinstance(fusion, str) else int(fusion)
        if kprime is None:
            kprime = limit * 3
        p = _Packed(self.dim, queries, sparse, None, None, limit, kprime, fz, sparse_weight, False)
        res, cres = self._alloc_result(p.B, limit, kprime, branches)
        self._check(self._lib.vb_merge_fuse(self._h, C.byref(p.c), int(n_shards), _vp(gathered_dev_ptr), C.byref(cres)))
        return res

    # ---- staged form (vb_stage / vb_run_local / vb_run_fuse / vb_fetch) -------------------------
    def stage(self, queries, sparse=None, filters=None, filter_of=None, limit: int = 10, kprime: int | None = None,
              fusion: str | int = "weighted", sparse_weight: float = 0.1, apply_idf: bool = True,
              branches: bool = False, need_corpus: bool = True):
        """Upload a batch; returns the (result, handle) pair that ``fetch`` fills."""
        fz = FUSION[fusion] if isinstance(fusion, str) else int(fusion)
        if kprime is None:
            kprime = limit * 3 if (sparse is not None and fz != FUSE_DENSE_ONLY) else limit
        p = _Packed(self.dim, queries, sparse, filters, filter_of, limit, kprime, fz, sparse_weight, apply_idf)
        if p.q_dev is not None:
            self._check(self._lib.vb_stage_dev(self._h, C.byref(p.c), p.q_dev.data_ptr(), p.q_stream, int(branches), int(need_corpus)))
        else:
            self._check(self._lib.vb_stage(self._h, C.byref(p.c), int(branches), int(need_corpus)))
        res, cres = self._alloc_result(p.B, limit, kprime, branches)
        return res, cres

    def stage_packed(self, packed, need_corpus: bool = True):
        """vb_stage on host buffers built earlier by ``pack`` (branches as chosen there)."""
        res, cres = packed.result
        want = res.dense_rows is not None
        if packed.q_dev is not None:
            self._check(self._lib.vb_stage_dev(self._h, C.byref(packed.c), packed.q_dev.data_ptr(), packed.q_stream, int(want), int(need_corpus)))
        else:
            self._check(self._lib.vb_stage(self._h, C.byref(packed.c), int(want), int(need_corpus)))
        return packed.result

    def run_local(self, cand_dev_ptr: int | None = None) -> None:
        self._check(self._lib.vb_run_local(self._h, _vp(cand_dev_ptr)))

    def run_fuse(self, n_shards: int = 0, gathered_dev_ptr: int | None = None) -> None:
        self._check(self._lib.vb_run_fuse(self._h, int(n_shards), _vp(gathered_dev_ptr)))

    def fetch(self, staged, allow_overflow: bool = False) -> SearchResult | None:
        """D2H + sync + decode.  Returns None (if allowed) when a candidate list overflowed and the
        staged batch must be re-run with set_option('safe_mode', 1)."""
        res, cres = staged
        ovf = C.c_int32()
        self._check(self._lib.vb_fetch(self._h, C.byref(cres), C.byref(ovf)))
        if ovf.value:
            if allow_overflow:
                return None
            raise B200Error("candidate list overflow: re-run with set_option('safe_mode', 1) or use search_batch")
        return res

    def set_option(self, key: str, value: int) -> None:
        self._check(self._lib.vb_set_option(self._h, key.encode(), int(value)))

    def stats(self) -> dict:
        s = _Stats()
        self._check(self._lib.vb_get_stats(self._h, C.byref(s)))
        return {k: getattr(s, k) for k, _ in _Stats._fields_}

    def timeline(self):
        """[(phase name, largest-launch flag, start ms, end ms)] of the last fetched search (option profile = 1)."""
        n = C.c_uint32()
        buf = np.zeros(3 * 4096, np.float64)
        self._check(self._lib.vb_get_timeline(self._h, _vp(buf), 4096, C.byref(n)))
        names = ["mask", "dense", "sparse", "select", "fuse"]
        return [(names[int(buf[3 * i]) & 7], bool(int(buf[3 * i]) & 8), float(buf[3 * i + 1]), float(buf[3 * i + 2]))
                for i in range(min(int(n.value), 4096))]

    def sync(self) -> None:
        self._check(self._lib.vb_sync(self._h))
