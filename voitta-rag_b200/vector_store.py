"""Drop-in replacement for ``voitta.services.vector_store`` backed by the B200 index.

Same names, argument order, defaults, return types and error behaviour as the reference class
(/root/reference/src/voitta/services/vector_store.py:18-1028): ``ChunkMetadata``, ``StoredChunk``,
``VectorStoreService`` (22 methods) and ``get_vector_store()``.  What the reference forwards to
Qdrant is split in two here:

  * arithmetic (cosine top-k, IDF sparse scoring, filter evaluation, fusion) -> the CUDA library
    through ``engine.Index`` (C ABI, include/voitta_b200.h);
  * payloads, point ids and the exact-match lookups behind the scroll / count / delete helpers ->
    host-side maps in ``_Collection`` (they are dictionary work, not GPU work; SURVEY.md §8 A10/A11).

State is process-global per collection name, so a second ``VectorStoreService()`` (as
api/routes/folders.py:139-141 creates) sees the same index.  Thread-safe (one re-entrant lock per
collection; callers are MCP worker threads, the indexing worker and the watchdog thread).

Additive API (not in the reference): ``search_batch``, ``search_visible`` (results restricted to the chunks a caller
may see, by each chunk's ``allowed_users``) and the ``fusion`` switch (``VOITTA_FUSION=weighted|rrf``; default
``weighted`` = the reference's behaviour).
"""
from __future__ import annotations

import atexit
import json
import logging
import os
from pathlib import Path
import threading
import time
import uuid
from dataclasses import dataclass

import numpy as np

from . import engine

logger = logging.getLogger("voitta.services.vector_store")

SPARSE_VECTOR_NAME = "bm25"  # reference: services/sparse_embedding.py:9


@dataclass
class ChunkMetadata:
    """Metadata for a stored chunk (reference :18-41)."""

    file_path: str
    folder_path: str
    index_folder: str
    file_name: str
    chunk_index: int
    total_chunks: int
    start_char: int
    end_char: int
    indexed_at: str
    start_page: int | None = None
    end_page: int | None = None
    source_page_count: int | None = None
    source_created_at: int | None = None
    source_modified_at: int | None = None
    allowed_users: list[str] | None = None
    source_url: str | None = None


@dataclass
class StoredChunk:
    """A chunk stored in the vector database (reference :44-51)."""

    id: str
    text: str
    metadata: ChunkMetadata
    score: float | None = None


class _Settings:
    """The six keys the reference store reads from voitta.config (config.py:28-34,44,72) plus
    the backend's own."""

    def __init__(self):
        self.qdrant_host = os.getenv("QDRANT_HOST", "localhost")
        self.qdrant_port = int(os.getenv("QDRANT_PORT", "6333"))
        self.qdrant_collection = os.getenv("QDRANT_COLLECTION", "voitta_documents")
        self.embedding_dimension = int(os.getenv("EMBEDDING_DIMENSION", "768"))
        self.device = int(os.getenv("VOITTA_B200_DEVICE", "0"))
        self.fusion = os.getenv("VOITTA_FUSION", "weighted")
        # directory of a snapshot to restore on first use (stands in for Qdrant's storage volume)
        self.snapshot_dir = os.getenv("VOITTA_B200_SNAPSHOT_DIR") or None
        # seconds between automatic snapshots after writes (unset = only save_snapshot() and the exit hook; the
        # reference persists every write through Qdrant, here a restart restores the last snapshot)
        a = os.getenv("VOITTA_B200_AUTOSAVE_SECS")
        self.autosave_secs = float(a) if a not in (None, "") else None


def get_settings() -> _Settings:
    return _Settings()


_OPTIONAL = ("start_page", "end_page", "source_page_count", "source_created_at",
             "source_modified_at", "allowed_users", "source_url")


def _principals(v, what: str) -> list[str]:
    """A list of principal strings (user e-mail, group ids).  A bare string is refused: iterating its characters
    would grant access by single letters."""
    if isinstance(v, (str, bytes)):
        raise TypeError(f"{what} must be a list of strings, not a single string")
    out = list(v)
    for p in out:
        if not isinstance(p, str):
            raise TypeError(f"{what} entries must be strings, got {type(p).__name__}")
    return out


def _acl_of(allowed_users) -> frozenset | None:
    """The ACL a row's ``allowed_users`` stands for: None = no ACL (visible to everyone), otherwise the set of
    principals that may see the row (empty = nobody)."""
    return None if allowed_users is None else frozenset(_principals(allowed_users, "allowed_users"))


def _is_device_tensor(x) -> bool:
    """A torch CUDA tensor (duck-typed: this module does not import torch)."""
    return bool(getattr(x, "is_cuda", False)) and hasattr(x, "data_ptr")


def _payload_to_chunk(pid: str, payload: dict, score) -> StoredChunk:
    """reference :532-558 (_result_to_chunk) and the identical blocks at :186-210, :943-965.
    Positional construction in dataclass field order: this runs 20 times per search on the caller's thread."""
    g = payload.get
    folder = payload["folder_path"]
    return StoredChunk(
        str(pid), payload["text"],
        ChunkMetadata(payload["file_path"], folder, g("index_folder", folder), payload["file_name"],
                      payload["chunk_index"], payload["total_chunks"], payload["start_char"], payload["end_char"],
                      payload["indexed_at"], g("start_page"), g("end_page"), g("source_page_count"),
                      g("source_created_at"), g("source_modified_at"), g("allowed_users"), g("source_url")),
        score)


class _Request:
    __slots__ = ("q", "sparse", "flt", "limit", "fusion", "sparse_weight", "done", "result", "error", "event", "lead")

    def __init__(self, q, sparse, flt, limit, fusion, sparse_weight):
        self.q, self.sparse, self.flt, self.limit, self.fusion, self.sparse_weight = q, sparse, flt, limit, fusion, sparse_weight
        self.done, self.result, self.error = False, None, None
        self.event = None            # created only when the request has to wait (a lone caller never does)
        self.lead = False            # set by the previous leader: "you run the next batch"


class _Coalescer:
    """Combines concurrent single-query searches into one device batch.

    voitta only ever issues B = 1 (mcp_server.py:474-485), but from several threads at once (FastMCP tool
    workers; SURVEY §8b).  Holding the collection lock for one device search per caller would serialise
    them at ~1 search latency each; instead the first caller to find the device free becomes the LEADER,
    takes every request queued so far — each with its own filter, the C ABI takes one filter per query —
    runs them as ONE vb_search, and hands the results back.  Callers that arrive while a batch is running
    queue up and form the next batch, so the batch size adapts to the load and a lone caller pays no wait.

    Hand-over is point to point: every waiter sleeps on its OWN event; a finishing leader wakes exactly the
    callers it served plus ONE queued caller, which becomes the next leader.  (The first version used one
    condition variable and notify_all: with 16 callers every batch woke 15 threads that fought for the GIL
    only to go back to sleep — 16 threads were SLOWER than one on small corpora, p99 170 ms.)"""

    def __init__(self, coll):
        self.coll = coll
        self.mu = threading.Lock()
        self.pending: list[_Request] = []
        self.busy = False
        self.batches = 0
        self.requests = 0

    def submit(self, req: _Request):
        with self.mu:
            if self.busy:
                req.event = threading.Event()
                self.pending.append(req)
                batch = None
            else:
                self.busy = True
                batch = [req]
        if batch is None:
            req.event.wait()
            if req.lead:                            # promoted by the previous leader: run everything queued so far
                with self.mu:
                    batch, self.pending = [req] + self.pending, []
        if batch is not None:
            try:
                self._run(batch)
            finally:
                with self.mu:
                    self.batches += 1
                    self.requests += len(batch)
                    nxt = self.pending.pop(0) if self.pending else None
                    if nxt is None:
                        self.busy = False
                    else:
                        nxt.lead = True             # busy stays set: the device is handed over, never released
                for r in batch:
                    if r is not req:
                        r.event.set()
                if nxt is not None:
                    nxt.event.set()
        if req.error is not None:
            raise req.error
        return req.result

    def _run(self, batch: list[_Request]):
        coll = self.coll
        groups: dict = {}
        for r in batch:                             # one device call per (limit, fusion, weight): the C ABI's per-batch knobs
            groups.setdefault((r.limit, r.fusion, r.sparse_weight), []).append(r)
        for (limit, fusion, weight), reqs in groups.items():
            try:
                with coll.lock:
                    if coll.n_live == 0:
                        for r in reqs:
                            r.result = []
                        continue
                    index = coll.index
                    flts, fo = [], []
                    for r in reqs:
                        if r.flt is None:
                            fo.append(-1)
                            continue
                        for i, f in enumerate(flts):
                            if f is r.flt:
                                fo.append(i)
                                break
                        else:
                            fo.append(len(flts))
                            flts.append(r.flt)
                    any_sparse = any(r.sparse is not None for r in reqs)
                    res = index.search_batch(
                        np.stack([r.q for r in reqs]), [r.sparse for r in reqs] if any_sparse else None,
                        filters=flts or None, filter_of=np.asarray(fo, np.int32) if flts else None,
                        limit=limit, kprime=limit * 3 if any_sparse else limit,
                        fusion=fusion if any_sparse else "dense", sparse_weight=weight)
                    base = getattr(index, "row_base", 0)
                    for i, r in enumerate(reqs):
                        r.result = [_payload_to_chunk(coll.ids[row - base], coll.payload[row - base], score) for row, score in res.hits(i)]
            except Exception as e:                  # every caller of the failed device call sees the error (reference: propagate)
                for r in reqs:
                    r.error = e
            finally:
                for r in reqs:
                    r.done = True


class _Collection:
    """Host half of one collection: ids, payloads and exact-match maps; owns the device index."""

    def __init__(self, name: str, dim: int, device: int, index_factory=None):
        self.name = name
        self.dim = dim
        self.device = device
        self.lock = threading.RLock()
        self._factory = index_factory or (lambda: engine.Index(dim, device=device))
        self._index = None
        self.ids: list[str] = []              # row -> point id
        self.payload: list[dict | None] = []  # row -> payload (None once deleted)
        self.n_live = 0
        self.by_file: dict[str, set[int]] = {}
        self.by_folder: dict[str, set[int]] = {}
        self.by_index_folder: dict[str, set[int]] = {}
        self.by_url: dict[str, set[int]] = {}
        # scope key -> scope id.  A key is (folder_path, index_folder) for rows without allowed_users and
        # (folder_path, index_folder, acl_id) for rows with them; acl_id indexes acl_list.
        self.scopes: dict[tuple, int] = {}
        self.scope_list: list[tuple] = []
        self.acl_list: list[frozenset] = []    # acl id -> the distinct allowed_users sets (frozenset() included)
        self.acl_ids: dict[frozenset, int] = {}
        self.scope_version = 0                 # bumped whenever a scope id is added: cached scope bitsets die with it
        self.bits_cache: dict = {}             # caller's scope_key -> (scope_version, args, bits)
        self._acl_fold = None                  # (scope_version, acl id + 1 per scope, principal -> acl ids + 1, any ACL)
        # set_file_acl met an index that cannot rewrite scope ids (no set_scope): its rows keep their old scope, so the
        # collection refuses visible_to from then on rather than answer from stale ids
        self.acl_stale = False
        self.coalescer = _Coalescer(self)
        self.dirty = False                     # written since the last snapshot
        self.last_save = time.monotonic()

    @property
    def index(self):
        with self.lock:
            if self._index is None:
                logger.info(f"Creating B200 index '{self.name}' (dim={self.dim}, device={self.device})")
                self._index = self._factory()
            return self._index

    def scope_id(self, folder_path: str, index_folder: str, acl: frozenset | None = None) -> int:
        if acl is None:
            key = (folder_path, index_folder)
        else:
            aid = self.acl_ids.get(acl)
            if aid is None:
                aid = self.acl_ids[acl] = len(self.acl_list)
                self.acl_list.append(acl)
            key = (folder_path, index_folder, aid)
        sid = self.scopes.get(key)
        if sid is None:
            sid = len(self.scope_list)
            self.scopes[key] = sid
            self.scope_list.append(key)
            self.scope_version += 1
        return sid

    def acl_fold(self):
        """What the ACL clause of a filter needs, rebuilt from scope_list / acl_list whenever scope_version changes:
        per scope its acl id + 1 (0 = unrestricted), per principal the acl ids + 1 that name it, and whether any
        scope carries an ACL.  Caller holds the lock."""
        f = self._acl_fold
        if f is None or f[0] != self.scope_version:
            scope_acl = np.fromiter((k[2] + 1 if len(k) > 2 else 0 for k in self.scope_list), np.int64, len(self.scope_list))
            by_principal: dict[str, list[int]] = {}
            for aid, acl in enumerate(self.acl_list):
                for p in acl:
                    by_principal.setdefault(p, []).append(aid + 1)
            f = self._acl_fold = (self.scope_version, scope_acl, {p: np.asarray(a, np.int64) for p, a in by_principal.items()},
                                  bool((scope_acl > 0).any()))
        return f

    def acl_bits(self, principals: list[str]):
        """Scope bitset of the rows visible to ``principals``, or None when every scope is (the clause drops out).
        Caller holds the lock."""
        _, scope_acl, by_principal, restricted = self.acl_fold()
        if not restricted:
            return None
        ok = np.zeros(len(self.acl_list) + 1, bool)
        ok[0] = True                                      # rows without allowed_users
        for p in principals:
            a = by_principal.get(p)
            if a is not None:
                ok[a] = True
        passing = ok[scope_acl]
        if passing.all():
            return None
        words = max(1, (len(passing) + 31) // 32)
        packed = np.zeros(words * 4, np.uint8)
        b = np.packbits(passing, bitorder="little")       # bit s of byte s / 8 = bit s of word s / 32 (little-endian words)
        packed[:len(b)] = b
        return packed.view("<u4").astype(np.uint32)

    def _map_add(self, m: dict, key, row: int):
        if key is not None:
            m.setdefault(key, set()).add(row)

    def add_rows(self, first_row: int, ids: list[str], payloads: list[dict]):
        if first_row != len(self.ids):
            raise RuntimeError(f"collection '{self.name}': device index has {first_row} rows, host maps {len(self.ids)} "
                               "(an earlier write failed half-way); reload the collection from its snapshot")
        for i, (pid, p) in enumerate(zip(ids, payloads)):
            r = first_row + i
            self.ids.append(pid)
            self.payload.append(p)
            self._map_add(self.by_file, p["file_path"], r)
            self._map_add(self.by_folder, p["folder_path"], r)
            self._map_add(self.by_index_folder, p["index_folder"], r)
            self._map_add(self.by_url, p.get("source_url"), r)
        self.n_live += len(ids)

    def remove_rows(self, rows: list[int]):
        for r in rows:
            p = self.payload[r]
            if p is None:
                continue
            for m, k in ((self.by_file, p["file_path"]), (self.by_folder, p["folder_path"]),
                         (self.by_index_folder, p["index_folder"]), (self.by_url, p.get("source_url"))):
                if k is not None and k in m:
                    m[k].discard(r)
                    if not m[k]:
                        del m[k]
            self.payload[r] = None
            self.n_live -= 1

    def live_rows(self):
        return (r for r, p in enumerate(self.payload) if p is not None)

    # ---- snapshot ---------------------------------------------------------------------------------
    # <dir>/<name>.<generation>.vb200   device data (vb_save)
    # <dir>/<name>.host.json            ids, payloads, scope dictionary + the generation it belongs to
    # The JSON file is the commit record: it is written last, to a temporary name, fsynced and renamed, and it
    # names the device file of the same generation — a crash at any point leaves the previous pair intact.
    # JSON, not pickle: the directory comes from the environment and must not be able to run code on load.
    def snapshot_paths(self, directory, generation: str | None = None):
        d = Path(directory)
        host = d / f"{self.name}.host.json"
        if generation is None and host.exists():
            try:
                with open(host, "r", encoding="utf-8") as f:
                    head = f.read(4096)
                generation = json.loads(head[:head.index(', "ids"')] + "}").get("generation")
            except Exception:
                generation = None
        return d / f"{self.name}.{generation or 'none'}.vb200", host

    def save(self, directory) -> dict:
        d = Path(directory)
        d.mkdir(parents=True, exist_ok=True)
        generation = uuid.uuid4().hex
        dev_path, host_path = self.snapshot_paths(d, generation)
        dev_tmp, host_tmp = dev_path.with_suffix(".vb200.tmp"), host_path.with_suffix(".json.tmp")
        with self.lock:
            self.index.save(dev_tmp)                       # vb_save flushes and fsyncs before it returns
            os.replace(dev_tmp, dev_path)
            # version 3 once a scope carries an ACL: a build that does not know ACLs refuses such a snapshot
            version = 3 if any(len(k) > 2 for k in self.scope_list) else 2
            head = {"version": version, "name": self.name, "dim": self.dim, "generation": generation,
                    "device_file": dev_path.name, "n_rows": len(self.ids), "n_live": self.n_live}
            if self.acl_stale:
                head["acl_stale"] = True
            with open(host_tmp, "w", encoding="utf-8") as f:
                # the small header keys come first so that snapshot_paths can read them without parsing the payloads
                f.write(json.dumps(head)[:-1] + ', "ids": ')
                json.dump(self.ids, f)
                f.write(', "scope_list": ')
                json.dump([list(k) for k in self.scope_list], f)
                f.write(', "acl_list": ')
                json.dump([sorted(a) for a in self.acl_list], f)
                f.write(', "payload": ')
                json.dump(self.payload, f)
                f.write("}")
                f.flush()
                os.fsync(f.fileno())
            os.replace(host_tmp, host_path)
            try:
                dfd = os.open(d, os.O_RDONLY)
                try:
                    os.fsync(dfd)
                finally:
                    os.close(dfd)
            except OSError:
                pass
            for old in d.glob(f"{self.name}.*.vb200"):     # device files of earlier generations
                if old != dev_path:
                    try:
                        old.unlink()
                    except OSError:
                        pass
            self.last_save = time.monotonic()
            self.dirty = False
        return {"rows": len(self.ids), "live": self.n_live, "device_file": str(dev_path), "host_file": str(host_path),
                "generation": generation}

    def load(self, directory, index_loader=None) -> int:
        """Replace this collection's contents with a snapshot.  Returns the number of live points."""
        d = Path(directory)
        _, host_path = self.snapshot_paths(d, "x")
        with open(host_path, "r", encoding="utf-8") as f:
            st = json.load(f)
        if st.get("version") not in (2, 3) or st.get("dim") != self.dim or st.get("name") != self.name:
            raise ValueError(f"snapshot {host_path} does not match collection '{self.name}' (dim {self.dim})")
        ids, payload = st["ids"], st["payload"]
        n_live = sum(1 for p in payload if p is not None)
        scope_list = [tuple(k) for k in st["scope_list"]]
        acl_list = [frozenset(a) for a in st.get("acl_list", [])]
        if any(len(k) not in (2, 3) or (len(k) == 3 and not 0 <= k[2] < len(acl_list)) for k in scope_list):
            raise ValueError(f"snapshot {host_path}: a scope names an ACL the snapshot does not hold")
        if len(ids) != len(payload) or len(ids) != st["n_rows"] or n_live != st["n_live"]:
            raise ValueError(f"snapshot {host_path} is inconsistent (ids {len(ids)}, payloads {len(payload)}, "
                             f"header rows {st['n_rows']} live {st['n_live']} / counted {n_live})")
        dev_path = d / st["device_file"]
        if Path(st["device_file"]).name != st["device_file"] or not dev_path.exists():
            raise ValueError(f"snapshot {host_path}: device file {st['device_file']} of generation {st.get('generation')} is missing")
        loader = index_loader or (lambda path: engine.Index.load(path, device=self.device))
        with self.lock:
            new_index = loader(dev_path)
            try:
                ist = new_index.stats()
                if int(ist["n_rows"]) != len(ids) or int(ist["n_live"]) != n_live or int(ist.get("dim", self.dim)) != self.dim:
                    raise ValueError(f"snapshot {host_path}: device file holds {ist['n_rows']} rows / {ist['n_live']} live "
                                     f"(dim {ist.get('dim')}), host file {len(ids)} / {n_live} (dim {self.dim})")
            except Exception:
                new_index.close()
                raise
            if self._index is not None:
                self._index.close()
            self._index = new_index
            self.ids = [str(x) for x in ids]
            self.payload = [None] * len(self.ids)
            self.n_live = 0
            self.by_file, self.by_folder, self.by_index_folder, self.by_url = {}, {}, {}, {}
            self.scope_list = scope_list
            self.scopes = {k: i for i, k in enumerate(self.scope_list)}
            self.acl_list = acl_list
            self.acl_ids = {a: i for i, a in enumerate(acl_list)}
            self.acl_stale = bool(st.get("acl_stale", False))
            self.scope_version += 1
            self.bits_cache.clear()
            for r, pl in enumerate(payload):
                if pl is None:
                    continue
                self.payload[r] = pl
                self._map_add(self.by_file, pl["file_path"], r)
                self._map_add(self.by_folder, pl["folder_path"], r)
                self._map_add(self.by_index_folder, pl["index_folder"], r)
                self._map_add(self.by_url, pl.get("source_url"), r)
                self.n_live += 1
            self.dirty = False
            self.last_save = time.monotonic()
            return self.n_live

    def wrote(self):
        """Called after every write (under the lock): autosave if VOITTA_B200_AUTOSAVE_SECS has elapsed."""
        self.dirty = True
        st = get_settings()
        if st.snapshot_dir and st.autosave_secs is not None and time.monotonic() - self.last_save >= st.autosave_secs:
            self.save(st.snapshot_dir)


_collections: dict[str, _Collection] = {}
_collections_lock = threading.Lock()


def _get_collection(name: str, dim: int, device: int, index_factory=None) -> _Collection:
    with _collections_lock:
        c = _collections.get(name)
        if c is None:
            c = _Collection(name, dim, device, index_factory)
            snap = get_settings().snapshot_dir
            if snap and index_factory is None and all(p.exists() for p in c.snapshot_paths(snap)):
                logger.info(f"Restoring collection '{name}' from {snap}")
                c.load(snap)
            if snap and index_factory is None:
                _register_exit_save()
            _collections[name] = c
        elif c.dim != dim:
            raise ValueError(f"collection '{name}' exists with dimension {c.dim}, requested {dim}")
        return c


_exit_hook = False


def _register_exit_save() -> None:
    """Save every collection written since its last snapshot when the process exits (the reference's
    Qdrant volume survives restarts; SQLite would otherwise claim files are indexed that are gone)."""
    global _exit_hook
    if _exit_hook:
        return
    _exit_hook = True

    def _save_all():
        snap = get_settings().snapshot_dir
        if not snap:
            return
        for c in list(_collections.values()):
            if c.dirty and c._index is not None:
                try:
                    c.save(snap)
                except Exception as e:       # pragma: no cover - best effort at exit
                    logger.error(f"exit snapshot of '{c.name}' failed: {e}")

    atexit.register(_save_all)


def _drop_collection(name: str) -> None:
    """Test helper: forget a collection (frees the device index)."""
    with _collections_lock:
        c = _collections.pop(name, None)
    if c is not None and c._index is not None:
        c._index.close()


class VectorStoreService:
    """Service for storing and retrieving document chunks on the B200 index (reference :54)."""

    def __init__(self, _index_factory=None):
        settings = get_settings()
        self.host = settings.qdrant_host
        self.port = settings.qdrant_port
        self.collection_name = settings.qdrant_collection
        self.dimension = settings.embedding_dimension
        self.fusion = settings.fusion
        self._device = settings.device
        self._client = None
        self._has_sparse: bool = False
        self._index_factory = _index_factory

    # ---- lazy "connection" (reference :66-115) --------------------------------------------------
    @property
    def _coll(self) -> _Collection:
        return _get_collection(self.collection_name, self.dimension, self._device, self._index_factory)

    @property
    def client(self):
        """Lazy-create the device index (the reference lazily connects to Qdrant here)."""
        if self._client is None:
            self._client = self._coll.index
            self._ensure_collection()
        return self._client

    def _ensure_collection(self) -> None:
        # a new collection always carries the sparse vector "bm25" with IDF (reference :95-99,114)
        self._has_sparse = True

    # ---- helpers --------------------------------------------------------------------------------
    def _rows_where(self, coll: _Collection, m: dict, key) -> list[int]:
        return sorted(r for r in m.get(key, ()) if coll.payload[r] is not None)

    def _by_id(self, coll: _Collection, rows) -> list[int]:
        """scroll() order: ascending point id."""
        return sorted(rows, key=lambda r: coll.ids[r])

    def find_by_source_url(self, source_url: str) -> list[StoredChunk]:
        """Find all chunks matching a given source_url, sorted by chunk_index (reference :163)."""
        coll = self._coll
        with coll.lock:
            rows = self._by_id(coll, self._rows_where(coll, coll.by_url, source_url))
            chunks = [_payload_to_chunk(coll.ids[r], coll.payload[r], None) for r in rows]
        chunks.sort(key=lambda c: c.metadata.chunk_index)
        return chunks

    def set_file_acl(self, file_path: str, allowed_users: list[str]) -> None:
        """Update allowed_users on all chunks for a specific file (reference :216).

        The rows move to the scope of their (folder, index folder, ACL) on the device first; the payloads change only
        once that succeeded, so a failed device call leaves both sides as they were.  An index without ``set_scope``
        gets the payload update only, and the collection then refuses ``visible_to`` (fails closed)."""
        acl = _acl_of(allowed_users)
        coll = self._coll
        with coll.lock:
            rows = self._rows_where(coll, coll.by_file, file_path)
            if not rows:
                return
            index = self.client
            if not hasattr(index, "set_scope"):
                # an index without vb_set_scope keeps the rows' scope ids: the payloads change as in the reference, and
                # the collection refuses visible_to from now on (_build_filter) instead of filtering by the old ACL
                for r in rows:
                    coll.payload[r]["allowed_users"] = allowed_users
                coll.acl_stale = True
                coll.wrote()
                return
            sids = np.fromiter((coll.scope_id(coll.payload[r]["folder_path"], coll.payload[r]["index_folder"], acl) for r in rows),
                               dtype=np.uint32, count=len(rows))
            index.set_scope(np.asarray(rows, dtype=np.uint64) + np.uint64(getattr(index, "row_base", 0)), sids)
            for r in rows:
                coll.payload[r]["allowed_users"] = allowed_users
            coll.wrote()

    def store_chunks(
        self,
        chunks: list[tuple[str, list[float], ChunkMetadata]],
        sparse_vectors: list[tuple[list[int], list[float]]] | None = None,
        batch_size: int = 100,
    ) -> list[str]:
        """Store multiple chunks with their embeddings; returns the generated point ids
        (reference :233-317)."""
        if not chunks:
            return []
        n = len(chunks)
        dense = np.empty((n, self.dimension), dtype=np.float32)
        ids, payloads = [], []
        indptr = np.zeros(n + 1, dtype=np.int64)
        terms, vals = [], []
        created = np.full(n, engine.TS_MISSING, dtype=np.int64)
        modified = np.full(n, engine.TS_MISSING, dtype=np.int64)
        coll = self._coll
        acls = []
        for idx, (text, embedding, metadata) in enumerate(chunks):
            acls.append(_acl_of(metadata.allowed_users))
            ids.append(str(uuid.uuid4()))
            payload = {
                "text": text,
                "file_path": metadata.file_path,
                "folder_path": metadata.folder_path,
                "index_folder": metadata.index_folder,
                "file_name": metadata.file_name,
                "chunk_index": metadata.chunk_index,
                "total_chunks": metadata.total_chunks,
                "start_char": metadata.start_char,
                "end_char": metadata.end_char,
                "indexed_at": metadata.indexed_at,
            }
            for k in _OPTIONAL:
                v = getattr(metadata, k)
                if v is not None:
                    payload[k] = v
            payloads.append(payload)
            if len(embedding) != self.dimension:
                raise ValueError(f"Vector dimension error: expected {self.dimension}, got {len(embedding)}")
            dense[idx] = embedding
            if metadata.source_created_at is not None:
                created[idx] = int(metadata.source_created_at)
            if metadata.source_modified_at is not None:
                modified[idx] = int(metadata.source_modified_at)
            nnz = 0
            if sparse_vectors and idx < len(sparse_vectors):
                indices, values = sparse_vectors[idx]
                if len(indices) != len(values):
                    raise ValueError("sparse vector indices/values length mismatch")
                if len(indices):
                    ix = np.asarray(indices, dtype=np.int64)
                    order = np.argsort(ix, kind="stable")   # qdrant sorts sparse vectors by index at upsert
                    ix = ix[order]
                    if (ix < 0).any() or (ix > 0xFFFFFFFF).any():
                        raise ValueError("sparse index out of uint32 range")
                    if (np.diff(ix) == 0).any():
                        raise ValueError("sparse vector indices must be unique")
                    terms.append(ix.astype(np.uint32))
                    vals.append(np.asarray(values, dtype=np.float32)[order])
                    nnz = len(ix)
            indptr[idx + 1] = indptr[idx] + nnz
        with coll.lock:
            scope = np.fromiter((coll.scope_id(p["folder_path"], p["index_folder"], a) for p, a in zip(payloads, acls)),
                                dtype=np.uint32, count=n)
            tcat = np.concatenate(terms) if terms else np.zeros(0, np.uint32)
            vcat = np.concatenate(vals) if vals else np.zeros(0, np.float32)
            index = self.client
            # One device upsert for the whole call (the C side chunks the H2D copies): either every row of
            # the call exists on both sides afterwards or none does.  The reference's batch_size (:311-313)
            # only sized its HTTP requests.
            first = index.upsert(dense, (indptr, tcat, vcat), scope, created, modified)
            try:
                coll.add_rows(first - getattr(index, "row_base", 0), ids, payloads)
            except Exception:
                # host bookkeeping failed after the device accepted the rows: tombstone them so that the two
                # sides keep the same live set, then surface the error
                index.delete_rows(np.arange(first, first + n, dtype=np.uint64))
                raise
            coll.wrote()
        logger.info(f"Stored {n} chunks in B200 index")
        return ids

    def _delete_where(self, m_name: str, key: str, what: str) -> int:
        coll = self._coll
        with coll.lock:
            rows = self._rows_where(coll, getattr(coll, m_name), key)
            count = len(rows)
            if count > 0:
                index = self.client
                base = getattr(index, "row_base", 0)
                index.delete_rows(np.asarray(rows, dtype=np.uint64) + np.uint64(base))
                coll.remove_rows(rows)
                coll.wrote()
                logger.info(f"Deleted {count} chunks for {what}: {key}")
        return count

    def delete_by_file(self, file_path: str) -> int:
        """Delete all chunks for a specific file; returns the number deleted (reference :319)."""
        return self._delete_where("by_file", file_path, "file")

    def delete_by_folder(self, folder_path: str) -> int:
        """Delete all chunks whose folder_path equals folder_path (reference :357)."""
        return self._delete_where("by_folder", folder_path, "folder")

    def delete_by_index_folder(self, index_folder: str) -> int:
        """Delete all chunks indexed from a specific index folder (reference :395)."""
        return self._delete_where("by_index_folder", index_folder, "index_folder")

    def get_file_paths_by_index_folder(self, index_folder: str) -> set[str]:
        """All unique file_path values for a given index_folder (reference :436)."""
        coll = self._coll
        with coll.lock:
            return {coll.payload[r]["file_path"] for r in self._rows_where(coll, coll.by_index_folder, index_folder)}

    # ---- filter (reference :462-530) ------------------------------------------------------------
    def _build_filter(
        self,
        folder_filter: str | None = None,
        include_folders: list[str] | None = None,
        exclude_folders: list[str] | None = None,
        exclude_index_folders: list[str] | None = None,
        date_start: int | None = None,
        date_end: int | None = None,
        date_field: str | None = None,
        scope_key=None,
        visible_to: list[str] | None = None,
    ) -> engine.Filter | None:
        """Evaluate the folder clauses over the scope dictionary and return the device filter.

        must folder_path == folder_filter; must folder_path IN include_folders (exact strings, the
        caller already expanded prefixes); must_not folder_path == e; must_not index_folder == f;
        must ts in [gte, lte] on source_created_at if date_field == "created" else source_modified_at.
        Returns None when no clause applies (reference :525-530).

        Additive: ``visible_to`` (a list of principals: the user's e-mail and group ids) keeps the rows whose
        ``allowed_users`` is absent or None, or shares an entry with it; ``allowed_users == []`` is visible to nobody.
        None adds no clause.  The clause is computed per call (the folder bits stay cached by ``scope_key``) and is
        left out when it passes every scope."""
        coll = self._coll
        if visible_to is not None:
            visible_to = _principals(visible_to, "visible_to")
            if coll.acl_stale:
                raise RuntimeError(f"collection '{coll.name}': an ACL changed on an index that cannot rewrite scope ids "
                                   "(no set_scope), so visible_to cannot be enforced")
        bits = None
        cached = None
        if scope_key is not None:
            # The caller (mcp_server.py:420-462) re-derives the same folder lists from SQLite for every query of a
            # (user, project); with a key that changes whenever those settings change, the folded bitset is reused
            # until a new scope (folder) appears in the collection.
            cached = coll.bits_cache.get(scope_key)
            if cached is not None and cached[0] != coll.scope_version:
                cached = None
        if cached is not None:
            bits = cached[1]
        elif folder_filter or include_folders or exclude_folders or exclude_index_folders:
            inc = set(include_folders) if include_folders else None
            exc = set(exclude_folders) if exclude_folders else ()
            dis = set(exclude_index_folders) if exclude_index_folders else ()
            with coll.lock:
                n_scopes = len(coll.scope_list)
                bits = np.zeros(max(1, (n_scopes + 31) // 32), dtype=np.uint32)
                for sid, key in enumerate(coll.scope_list):
                    fp, ifp = key[0], key[1]
                    ok = ((not folder_filter or fp == folder_filter) and (inc is None or fp in inc)
                          and fp not in exc and ifp not in dis)
                    if ok:
                        bits[sid >> 5] |= np.uint32(1 << (sid & 31))
                if scope_key is not None:
                    if len(coll.bits_cache) >= 256:
                        coll.bits_cache.pop(next(iter(coll.bits_cache)))
                    coll.bits_cache[scope_key] = (coll.scope_version, bits)
        if visible_to is not None:
            with coll.lock:
                acl = coll.acl_bits(visible_to)
            if acl is not None:
                if bits is None:
                    bits = acl
                else:                                     # a cached fold may predate scopes added since: they read as 0
                    n = min(len(bits), len(acl))
                    both = np.zeros(max(len(bits), len(acl)), np.uint32)
                    both[:n] = bits[:n] & acl[:n]
                    bits = both
        ts_field, lo, hi = engine.TS_NONE, engine.TS_MIN, engine.TS_MAX
        if date_start is not None or date_end is not None:
            field_map = {"created": engine.TS_CREATED, "modified": engine.TS_MODIFIED}
            ts_field = field_map.get(date_field, engine.TS_MODIFIED) if date_field else engine.TS_MODIFIED
            if date_start is not None:
                lo = max(engine.TS_MIN, int(np.ceil(date_start)))
            if date_end is not None:
                hi = min(engine.TS_MAX, int(np.floor(date_end)))
        if bits is None and ts_field == engine.TS_NONE:
            return None
        return engine.Filter(scope_bits=bits, ts_field=ts_field, ts_lo=lo, ts_hi=hi)

    def _rows_to_chunks(self, coll: _Collection, hits) -> list[StoredChunk]:
        base = getattr(coll.index, "row_base", 0)
        out = []
        for row, score in hits:
            r = row - base
            out.append(_payload_to_chunk(coll.ids[r], coll.payload[r], score))
        return out

    def search(
        self,
        query_embedding: list[float],
        limit: int = 10,
        folder_filter: str | None = None,
        include_folders: list[str] | None = None,
        exclude_folders: list[str] | None = None,
        exclude_index_folders: list[str] | None = None,
        sparse_query: tuple[list[int], list[float]] | None = None,
        sparse_weight: float = 0.1,
        date_start: int | None = None,
        date_end: int | None = None,
        date_field: str | None = None,
        scope_key=None,
    ) -> list[StoredChunk]:
        """Dense or hybrid (dense + sparse) retrieval (reference :560-697).

        Hybrid iff ``sparse_query`` has indices and the collection has the sparse vector: both
        branches fetch limit*3 candidates under the same filter and are fused (min-max weighted
        sum by default).  Otherwise dense-only with ``limit``.

        Additive: ``scope_key`` (any hashable, e.g. ``(user_id, project_id, settings_version)``) lets the
        folded folder bitset be cached across calls.  Concurrent callers are coalesced into one device
        batch (``_Coalescer``)."""
        return self._search(query_embedding, limit, folder_filter, include_folders, exclude_folders, exclude_index_folders,
                            sparse_query, sparse_weight, date_start, date_end, date_field, scope_key, None)

    def search_visible(
        self,
        query_embedding: list[float],
        limit: int = 10,
        folder_filter: str | None = None,
        include_folders: list[str] | None = None,
        exclude_folders: list[str] | None = None,
        exclude_index_folders: list[str] | None = None,
        sparse_query: tuple[list[int], list[float]] | None = None,
        sparse_weight: float = 0.1,
        date_start: int | None = None,
        date_end: int | None = None,
        date_field: str | None = None,
        scope_key=None,
        *,
        visible_to: list[str] | None,
    ) -> list[StoredChunk]:
        """Additive: ``search`` restricted to the chunks the caller may see.  ``visible_to`` lists the caller's
        principals (the user's e-mail plus the group ids the caller resolved); a chunk is returned only if its
        ``allowed_users`` is absent or None, or shares an entry with ``visible_to`` (see ``_build_filter``)."""
        return self._search(query_embedding, limit, folder_filter, include_folders, exclude_folders, exclude_index_folders,
                            sparse_query, sparse_weight, date_start, date_end, date_field, scope_key, visible_to)

    def _search(self, query_embedding, limit, folder_filter, include_folders, exclude_folders, exclude_index_folders,
                sparse_query, sparse_weight, date_start, date_end, date_field, scope_key, visible_to):
        self.client
        coll = self._coll
        if _is_device_tensor(query_embedding):
            # additive: a CUDA tensor from the embedding model goes to the device search as it is (no .tolist() hop)
            if query_embedding.dim() != 1 or query_embedding.shape[0] != self.dimension:
                raise ValueError(f"Vector dimension error: expected {self.dimension}, got {query_embedding.shape[-1] if query_embedding.dim() else 0}")
            return self.search_batch(query_embedding[None, :], limit=limit, folder_filter=folder_filter, include_folders=include_folders,
                                     exclude_folders=exclude_folders, exclude_index_folders=exclude_index_folders,
                                     sparse_queries=[sparse_query], sparse_weight=sparse_weight, date_start=date_start,
                                     date_end=date_end, date_field=date_field, visible_to=visible_to)[0]
        search_filter = self._build_filter(
            folder_filter, include_folders, exclude_folders, exclude_index_folders,
            date_start=date_start, date_end=date_end, date_field=date_field, scope_key=scope_key, visible_to=visible_to)
        q = np.asarray(query_embedding, dtype=np.float32)
        if q.ndim != 1 or q.shape[0] != self.dimension:
            raise ValueError(f"Vector dimension error: expected {self.dimension}, got {q.shape[-1] if q.ndim else 0}")
        if not np.isfinite(q).all():
            raise ValueError("Query vector must not contain NaN or inf")
        sparse = None
        if sparse_query and self._has_sparse:                  # reference :599-601
            indices, values = sparse_query
            if len(indices):
                sparse = (indices, values)
        return coll.coalescer.submit(_Request(q, sparse, search_filter, limit, self.fusion, sparse_weight))

    def _hybrid_search(self, query_embedding, sparse_query, limit=10, search_filter=None, sparse_weight=0.1):
        """Reference :621-697 (private there, no external callers): hybrid search with a prepared filter."""
        return self._coll.coalescer.submit(_Request(np.asarray(query_embedding, dtype=np.float32), sparse_query, search_filter,
                                                   limit, self.fusion, sparse_weight))

    def _result_to_chunk(self, result) -> StoredChunk:
        """Reference :532-558: anything with .id / .payload / .score (a qdrant ScoredPoint there)."""
        return _payload_to_chunk(result.id, result.payload, getattr(result, "score", None))

    def qdrant_facade(self) -> "QdrantScrollFacade":
        """Additive: a QdrantClient-shaped object for scripts/sync_qdrant_stats.py (get_collection + scroll)."""
        self.client
        return QdrantScrollFacade(self)

    def coalescing_stats(self) -> dict:
        """Device batches formed out of concurrent single-query searches so far."""
        c = self._coll.coalescer
        return {"batches": c.batches, "requests": c.requests, "mean_batch": (c.requests / c.batches) if c.batches else None}

    def search_batch(
        self,
        query_embeddings,
        limit: int = 10,
        folder_filter: str | None = None,
        include_folders: list[str] | None = None,
        exclude_folders: list[str] | None = None,
        exclude_index_folders: list[str] | None = None,
        sparse_queries=None,
        sparse_weight: float = 0.1,
        date_start: int | None = None,
        date_end: int | None = None,
        date_field: str | None = None,
        fusion: str | None = None,
        filters: list[dict | None] | None = None,
        visible_to: list[str] | None = None,
    ) -> list[list[StoredChunk]]:
        """Additive: ``search`` for B queries in one device pass.

        By default the B queries share one filter, built from the folder and date arguments.  ``filters`` gives each
        query its own instead: a list of B entries, each None (unfiltered) or a dict of ``_build_filter`` keyword
        arguments (``folder_filter``, ``include_folders``, ``exclude_folders``, ``exclude_index_folders``,
        ``date_start``, ``date_end``, ``date_field``, ``scope_key``, ``visible_to``).  Queries whose filters have equal
        content share one device mask.  Giving ``filters`` together with any of the shared filter arguments
        (``visible_to`` included) is a ValueError.  ``visible_to`` restricts the results to the chunks those principals
        may see, as in ``search_visible``."""
        index = self.client
        coll = self._coll
        B = len(query_embeddings)
        if filters is None:
            search_filter = self._build_filter(
                folder_filter, include_folders, exclude_folders, exclude_index_folders,
                date_start=date_start, date_end=date_end, date_field=date_field, visible_to=visible_to)
            flts = [search_filter] if search_filter is not None else None
            filter_of = np.zeros(B, np.int32) if search_filter is not None else None
        else:
            shared = (folder_filter, include_folders, exclude_folders, exclude_index_folders, date_start, date_end, date_field,
                      visible_to)
            if any(a is not None for a in shared):
                raise ValueError("give either per-query filters or the shared filter arguments, not both")
            if len(filters) != B:
                raise ValueError(f"filters must have one entry per query: {len(filters)} for {B} queries")
            flts, fo = [], np.full(B, -1, np.int32)
            for i, kw in enumerate(filters):
                f = None if kw is None else self._build_filter(**kw)
                if f is not None:
                    fo[i] = len(flts)
                    flts.append(f)
            filter_of = fo if flts else None
            flts = flts or None
        if _is_device_tensor(query_embeddings):
            # tensor hand-off (SURVEY 8 f-4): the embedding model's output (embedding.py:76-86) stays on the GPU
            q = query_embeddings
            if q.dim() != 2 or q.shape[1] != self.dimension:
                raise ValueError(f"Vector dimension error: expected {self.dimension}, got {q.shape[-1] if q.dim() else 0}")
        else:
            q = np.asarray(query_embeddings, dtype=np.float32)
            if q.ndim != 2 or q.shape[1] != self.dimension:
                raise ValueError(f"Vector dimension error: expected {self.dimension}, got {q.shape[-1] if q.ndim else 0}")
        sparse = [None] * B
        any_sparse = False
        if sparse_queries is not None and self._has_sparse:
            for i, sq in enumerate(sparse_queries):
                if sq:
                    indices, values = sq
                    if len(indices):
                        sparse[i] = (indices, values)
                        any_sparse = True
        with coll.lock:
            if coll.n_live == 0:
                return [[] for _ in range(B)]
            res = index.search_batch(
                q, sparse if any_sparse else None, filters=flts, filter_of=filter_of,
                limit=limit, kprime=limit * 3 if any_sparse else limit,
                fusion=(fusion or self.fusion) if any_sparse else "dense", sparse_weight=sparse_weight)
            return [self._rows_to_chunks(coll, res.hits(i)) for i in range(B)]

    # ---- collection / scroll helpers (reference :699-1016) --------------------------------------
    # ---- persistence (additive: the reference relies on Qdrant's storage volume) --------------------
    def save_snapshot(self, directory: str | None = None) -> dict:
        """Write the collection (device index + ids/payloads) under ``directory``
        (default: $VOITTA_B200_SNAPSHOT_DIR).  A process started with that variable set restores it
        on first use."""
        directory = directory or get_settings().snapshot_dir
        if not directory:
            raise ValueError("no snapshot directory given and VOITTA_B200_SNAPSHOT_DIR is not set")
        return self._coll.save(directory)

    def load_snapshot(self, directory: str | None = None, _index_loader=None) -> int:
        """Replace the collection's contents with the snapshot under ``directory``; returns live points."""
        directory = directory or get_settings().snapshot_dir
        if not directory:
            raise ValueError("no snapshot directory given and VOITTA_B200_SNAPSHOT_DIR is not set")
        n = self._coll.load(directory, _index_loader)
        self._client = self._coll.index
        self._ensure_collection()
        return n

    def get_collection_info(self) -> dict:
        """Information about the collection (reference :699)."""
        try:
            coll = self._coll
            return {
                "name": self.collection_name,
                "vectors_count": coll.n_live,
                "points_count": coll.n_live,
                "status": "green",
            }
        except Exception as e:
            return {"error": str(e)}

    def count_by_file(self, file_path: str) -> int:
        """Count chunks for a specific file (reference :712)."""
        try:
            coll = self._coll
            with coll.lock:
                return len(self._rows_where(coll, coll.by_file, file_path))
        except Exception:
            return 0

    def count_chunks_for_files(self, file_paths: list[str]) -> dict[str, int]:
        """Chunk counts for several files; only files with chunks appear (reference :730)."""
        if not file_paths:
            return {}
        try:
            coll = self._coll
            out: dict[str, int] = {}
            with coll.lock:
                for fp in dict.fromkeys(file_paths):
                    c = len(self._rows_where(coll, coll.by_file, fp))
                    if c:
                        out[fp] = c
            return out
        except Exception as e:
            logger.error(f"Error counting chunks for files: {e}")
            return {}

    def _file_counts(self, coll: _Collection) -> dict[str, int]:
        return {fp: n for fp, rows in coll.by_file.items() if (n := sum(1 for r in rows if coll.payload[r] is not None))}

    def count_chunks_for_folder(self, folder_path: str) -> tuple[int, int]:
        """(indexed file count, total chunk count) under a folder, recursively (reference :777)."""
        try:
            prefix = folder_path + "/" if folder_path else ""
            coll = self._coll
            with coll.lock:
                fc = {fp: n for fp, n in self._file_counts(coll).items()
                      if fp.startswith(prefix) or (not prefix and "/" not in fp)}
            return len(fc), sum(fc.values())
        except Exception as e:
            logger.error(f"Error counting chunks for folder {folder_path}: {e}")
            return 0, 0

    def get_folder_stats_batch(self, folder_paths: list[str]) -> dict[str, tuple[int, int]]:
        """(file count, chunk count) for several folders in one scan (reference :816)."""
        if not folder_paths:
            return {}
        try:
            coll = self._coll
            with coll.lock:
                counts = self._file_counts(coll)
            out = {}
            for folder in folder_paths:
                prefix = folder + "/" if folder else ""
                sel = [n for fp, n in counts.items() if fp.startswith(prefix) or (not prefix and "/" not in fp)]
                out[folder] = (len(sel), sum(sel))
            return out
        except Exception as e:
            logger.error(f"Error getting folder stats batch: {e}")
            return {fp: (0, 0) for fp in folder_paths}

    def get_stored_page_count(self, file_path: str) -> int | None:
        """Stored source_page_count of (any chunk of) a PDF file (reference :869)."""
        try:
            coll = self._coll
            with coll.lock:
                rows = self._by_id(coll, self._rows_where(coll, coll.by_file, file_path))
                if rows and coll.payload[rows[0]].get("source_page_count"):
                    return coll.payload[rows[0]]["source_page_count"]
            return None
        except Exception as e:
            logger.error(f"Error getting stored page count for {file_path}: {e}")
            return None

    def get_chunks_by_range(self, file_path: str, first_chunk: int, last_chunk: int) -> list[StoredChunk]:
        """Chunks of a file with first_chunk <= chunk_index <= last_chunk, sorted (reference :898)."""
        try:
            coll = self._coll
            with coll.lock:
                rows = self._by_id(coll, self._rows_where(coll, coll.by_file, file_path))
                chunks = [_payload_to_chunk(coll.ids[r], coll.payload[r], None) for r in rows
                          if first_chunk <= coll.payload[r]["chunk_index"] <= last_chunk]
            chunks.sort(key=lambda c: c.metadata.chunk_index)
            return chunks
        except Exception as e:
            logger.error(f"Error getting chunks by range for {file_path}: {e}")
            return []

    def get_file_chunk_counts(self, folder_prefix: str = "") -> dict[str, int]:
        """Chunk counts for all files, optionally restricted to a path prefix (reference :979)."""
        try:
            coll = self._coll
            with coll.lock:
                return {fp: n for fp, n in self._file_counts(coll).items()
                        if not folder_prefix or fp.startswith(folder_prefix)}
        except Exception as e:
            logger.error(f"Error getting file chunk counts: {e}")
            return {}


class _ScrollRecord:
    """What QdrantClient.scroll returns per point, as far as the reference's scripts read it: .id and .payload."""
    __slots__ = ("id", "payload")

    def __init__(self, pid, payload):
        self.id, self.payload = pid, payload


class _CollectionInfo:
    __slots__ = ("points_count",)

    def __init__(self, n):
        self.points_count = n


class QdrantScrollFacade:
    """The two QdrantClient calls of scripts/sync_qdrant_stats.py:29-81 (the admin script that rebuilds SQLite's
    indexed_files table from the vector store) over this backend's host-side payload store:
    ``get_collection(name).points_count`` and ``scroll(collection_name, limit, offset, with_payload, with_vectors)``
    -> ``(records, next_offset)``.  The script's only change is its client line:
    ``client = get_vector_store().qdrant_facade()`` instead of ``QdrantClient(host=..., port=...)``.
    Offsets are opaque to the caller (there: a point id; here: the next row), ``None`` ends the scan; deleted rows
    are skipped; ``with_payload`` may be True or a list of keys."""

    def __init__(self, store: "VectorStoreService"):
        self._store = store

    def _coll_for(self, collection_name):
        if collection_name not in (None, self._store.collection_name):
            raise ValueError(f"Collection {collection_name} not found")
        return self._store._coll

    def get_collection(self, collection_name=None):
        coll = self._coll_for(collection_name)
        with coll.lock:
            return _CollectionInfo(coll.n_live)

    def scroll(self, collection_name=None, scroll_filter=None, limit: int = 10, offset=None, with_payload=True, with_vectors=False):
        if scroll_filter is not None or with_vectors:
            raise NotImplementedError("the facade serves the unfiltered payload scan of sync_qdrant_stats.py")
        coll = self._coll_for(collection_name)
        out = []
        with coll.lock:
            r = int(offset or 0)
            n = len(coll.ids)
            while r < n and len(out) < limit:
                pl = coll.payload[r]
                if pl is not None:
                    if with_payload is True:
                        view = dict(pl)
                    elif with_payload:
                        view = {k: pl[k] for k in with_payload if k in pl}
                    else:
                        view = None
                    out.append(_ScrollRecord(coll.ids[r], view))
                r += 1
            while r < n and coll.payload[r] is None:           # do not hand out an offset that only leads to deleted rows
                r += 1
            return out, (r if r < n else None)


# Global singleton instance (reference :1019-1028)
_vector_store: VectorStoreService | None = None


def get_vector_store() -> VectorStoreService:
    """Get the global vector store service instance."""
    global _vector_store
    if _vector_store is None:
        _vector_store = VectorStoreService()
    return _vector_store
