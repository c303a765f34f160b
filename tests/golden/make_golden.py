#!/usr/bin/env python3
"""Generate tests/golden/voitta_cases.json by running the REFERENCE's own
``voitta/services/vector_store.py`` (unmodified, from the voitta-rag checkout that
$VOITTA_REFERENCE_SRC names).

``qdrant_client`` is not installable here (no network), so it is replaced by a stub whose
``QdrantClient`` delegates to ``oracle.oracle.LocalCollection`` (the restatement of
qdrant-client local mode).  Everything voitta owns on the path therefore runs as the
reference wrote it: point construction (:233-317), ``_build_filter`` (:462-530), the
``search`` dispatch (:560-619), min-max weighted fusion (:621-697), ``_result_to_chunk``
(:532-558), deletes / counts / scroll helpers.  The recorded outputs pin
``oracle.OracleVectorStore`` (tests/test_oracle_golden.py) and are replayed against the
B200 backend (tests/test_gpu_golden.py).

Run from the repo root:  VOITTA_REFERENCE_SRC=<voitta-rag>/src/voitta python tests/golden/make_golden.py
The reference source is NOT needed at test time; only this script reads it.
"""
from __future__ import annotations

import importlib.util
import json
import os
import sys
import types
import uuid
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

from oracle import oracle as O  # noqa: E402
import _data  # noqa: E402

DIM = 32
N = 600


# ----------------------------------------------------------------------------- stub qdrant_client
class _Enum:
    def __init__(self, value):
        self.value = value


class _NS(types.SimpleNamespace):
    pass


def _install_stub(dim_holder):
    qc = types.ModuleType("qdrant_client")
    http = types.ModuleType("qdrant_client.http")
    models = types.ModuleType("qdrant_client.http.models")
    exc = types.ModuleType("qdrant_client.http.exceptions")

    class UnexpectedResponse(Exception):
        pass

    exc.UnexpectedResponse = UnexpectedResponse
    models.Filter = O.Filter
    models.FieldCondition = O.FieldCondition
    models.MatchValue = O.MatchValue
    models.MatchAny = O.MatchAny
    models.Range = O.Range
    models.SparseVector = O.SparseVector
    models.Distance = _NS(COSINE="Cosine")
    models.Modifier = _NS(IDF="idf")
    models.PayloadSchemaType = _NS(KEYWORD="keyword", INTEGER="integer")
    models.VectorParams = lambda size, distance: _NS(size=size, distance=distance)
    models.SparseVectorParams = lambda modifier=None: _NS(modifier=modifier)
    models.PointStruct = lambda id, vector, payload: _NS(id=id, vector=vector, payload=payload)
    models.FilterSelector = lambda filter: _NS(filter=filter)

    class QdrantClient:
        """Only the nine methods vector_store.py calls."""

        def __init__(self, host=None, port=None, **kw):
            self.coll = None

        def get_collection(self, name):
            if self.coll is None:
                raise UnexpectedResponse("not found")
            return _NS(config=_NS(params=_NS(sparse_vectors={"bm25": 1} if self.coll.has_sparse else {})),
                       payload_schema={}, vectors_count=None,
                       points_count=self.coll.count(None), status=_Enum("green"))

        def create_collection(self, collection_name, vectors_config, sparse_vectors_config=None):
            assert vectors_config.distance == "Cosine"
            self.coll = O.LocalCollection(vectors_config.size, has_sparse=bool(sparse_vectors_config))

        def create_payload_index(self, **kw):
            pass

        def upsert(self, collection_name, points):
            for p in points:
                if isinstance(p.vector, dict):
                    sv = p.vector.get("bm25")
                    self.coll.upsert(p.id, p.vector[""], (sv.indices, sv.values) if sv else None, p.payload)
                else:
                    self.coll.upsert(p.id, p.vector, None, p.payload)

        def query_points(self, collection_name, query, limit, query_filter=None, using=None):
            if isinstance(query, O.SparseVector):
                assert using == "bm25"
                pts = self.coll.query_sparse(query.indices, query.values, limit, query_filter)
            else:
                pts = self.coll.query_dense(query, limit, query_filter)
            return _NS(points=pts)

        def scroll(self, collection_name, limit=10, offset=None, scroll_filter=None,
                   with_payload=True, with_vectors=False):
            return self.coll.scroll(scroll_filter, limit=limit, offset=offset)

        def count(self, collection_name, count_filter=None):
            return _NS(count=self.coll.count(count_filter))

        def delete(self, collection_name, points_selector):
            self.coll.delete(points_selector.filter)

        def set_payload(self, collection_name, payload, points):
            self.coll.set_payload(payload, points.filter)

    qc.QdrantClient = QdrantClient
    qc.http = http
    http.models = models
    http.exceptions = exc
    sys.modules.update({"qdrant_client": qc, "qdrant_client.http": http,
                        "qdrant_client.http.models": models, "qdrant_client.http.exceptions": exc})


def real_qdrant_available() -> bool:
    """True if the REAL qdrant-client can be imported (from the environment or from baseline/_ref, where a
    driver-provided reference install would land).  It is not part of this image; the probe runs every round."""
    ref_dir = ROOT / "baseline" / "_ref"
    if ref_dir.is_dir() and str(ref_dir) not in sys.path:
        sys.path.insert(0, str(ref_dir))
    mod = sys.modules.get("qdrant_client")
    if mod is not None and getattr(mod, "__file__", None) is None:
        return False                                   # our own stub is installed in this process
    try:
        return importlib.util.find_spec("qdrant_client") is not None
    except Exception:
        return False


def reference_src() -> Path | None:
    """voitta-rag's ``src/voitta`` directory, named by $VOITTA_REFERENCE_SRC; None if unset or not a checkout."""
    p = os.environ.get("VOITTA_REFERENCE_SRC")
    return Path(p) if p and (Path(p) / "services" / "vector_store.py").is_file() else None


def _install_real():
    """Route the reference's QdrantClient(host, port) to qdrant-client's local in-memory mode."""
    import qdrant_client
    real = qdrant_client.QdrantClient

    def local_client(host=None, port=None, **kw):
        return real(":memory:")

    qdrant_client.QdrantClient = local_client


def load_reference_vector_store(dim: int, real: bool = False):
    """Import the reference's services/vector_store.py (``reference_src()``) without running the
    package __init__ files (they import sqlalchemy/fastmcp/... which are absent).  ``real``: over the real
    qdrant-client (local mode) instead of the stub that delegates to the oracle."""
    REF = reference_src()
    if REF is None:
        raise RuntimeError("set VOITTA_REFERENCE_SRC to voitta-rag's src/voitta directory")
    if real:
        _install_real()
    else:
        _install_stub(dim)
    voitta = types.ModuleType("voitta"); voitta.__path__ = [str(REF)]
    services = types.ModuleType("voitta.services"); services.__path__ = [str(REF / "services")]
    config = types.ModuleType("voitta.config")
    settings = _NS(qdrant_host="stub", qdrant_port=0, qdrant_collection="golden", embedding_dimension=dim)
    config.get_settings = lambda: settings
    sys.modules.update({"voitta": voitta, "voitta.services": services, "voitta.config": config})
    for name in ("sparse_embedding", "vector_store"):
        spec = importlib.util.spec_from_file_location(f"voitta.services.{name}", REF / "services" / f"{name}.py")
        mod = importlib.util.module_from_spec(spec)
        sys.modules[spec.name] = mod
        spec.loader.exec_module(mod)
    return sys.modules["voitta.services.vector_store"]


# ----------------------------------------------------------------------------- the scenario
def scenario(corpus, queries):
    """The operation sequence replayed by the golden generator, the oracle test and the GPU
    test.  Rows are referred to by insertion index.  Covers SURVEY.md §8(c) items (i)-(xi)."""
    folders = [f for f, _ in corpus["folders"]]
    ops = []
    # ingest in 4 calls; the 3rd WITHOUT sparse vectors (rows lacking "bm25"), custom batch_size
    cuts = [0, 200, 400, 450, N]
    ops.append({"op": "store", "lo": cuts[0], "hi": cuts[1], "sparse": True})
    ops.append({"op": "store", "lo": cuts[1], "hi": cuts[2], "sparse": True, "batch_size": 37})
    ops.append({"op": "store", "lo": cuts[2], "hi": cuts[3], "sparse": False})
    ops.append({"op": "store", "lo": cuts[3], "hi": cuts[4], "sparse": True})
    ops.append({"op": "info"})

    def S(qi, **kw):
        ops.append({"op": "search", "q": qi, "kw": kw})

    for qi in range(6):                                      # (i) plain dense / hybrid
        S(qi, limit=10, sparse=False)
        S(qi, limit=10, sparse=True)
    S(0, limit=5, sparse=True, sparse_weight=0.0)
    S(0, limit=5, sparse=True, sparse_weight=0.5)
    S(1, limit=5, sparse=True, sparse_weight=0.9)
    S(1, limit=5, sparse=True, sparse_weight=1.0)
    S(2, limit=20, sparse=True)                              # MCP default limit (k'=60)
    S(2, limit=10, sparse="empty")                           # (viii) ([],[]) -> dense-only
    S(3, limit=10, sparse=True, folder_filter=folders[1])    # legacy single folder
    S(3, limit=10, sparse=True, include_folders=folders[:4])
    S(3, limit=10, sparse=False, include_folders=[folders[0]])
    S(3, limit=10, sparse=True, include_folders=[])          # [] == no include clause (:484)
    S(4, limit=10, sparse=True, exclude_folders=[folders[0], folders[5]])
    S(4, limit=10, sparse=True, exclude_index_folders=["root0"])
    S(4, limit=10, sparse=True, include_folders=folders[:8], exclude_folders=[folders[2]],
      exclude_index_folders=["root1"])
    S(5, limit=10, sparse=True, date_start=1500000000)                        # (vi) missing modified fails
    S(5, limit=10, sparse=True, date_end=1600000000)
    S(5, limit=10, sparse=True, date_start=1500000000, date_end=1650000000, date_field="created")  # (vii)
    S(5, limit=10, sparse=True, date_start=1500000000, date_end=1650000000, date_field="modified")
    S(5, limit=10, sparse=True, date_start=1500000000, date_end=1650000000, date_field="bogus")
    S(5, limit=10, sparse=False, date_start=1766000000, date_end=1767225600)  # very selective
    S(6, limit=10, sparse=True, include_folders=["no/such/folder"])           # nothing passes
    S(7, limit=10, sparse="rare")                            # (iv) sparse list shorter than k'
    S(7, limit=10, sparse="single")                          # (iii) one sparse hit -> spread == 0
    S(8, limit=200, sparse=True)                             # k' = 600 >= N: whole corpus ranked
    S(9, limit=3, sparse="absent")                           # term not in corpus: empty sparse list
    S(10, limit=10, sparse=True)                             # (ii) query == duplicated row
    # helpers
    m0 = corpus["metas"][0]
    ops.append({"op": "count_by_file", "arg": m0["file_path"]})
    ops.append({"op": "count_by_file", "arg": "nope"})
    ops.append({"op": "get_chunks_by_range", "args": [m0["file_path"], 1, 2]})
    urls = [m["source_url"] for m in corpus["metas"] if m["source_url"]]
    ops.append({"op": "find_by_source_url", "arg": urls[0]})
    ops.append({"op": "find_by_source_url", "arg": "https://nope"})
    pdfs = [m["file_path"] for m in corpus["metas"] if m["source_page_count"]]
    ops.append({"op": "get_stored_page_count", "arg": pdfs[0]})
    ops.append({"op": "get_stored_page_count", "arg": m0["file_path"] if not m0["source_page_count"] else "nope"})
    ops.append({"op": "get_file_paths_by_index_folder", "arg": "root1"})
    ops.append({"op": "count_chunks_for_files", "arg": [m0["file_path"], corpus["metas"][50]["file_path"], "nope"]})
    ops.append({"op": "count_chunks_for_folder", "arg": "root0"})
    ops.append({"op": "count_chunks_for_folder", "arg": ""})
    ops.append({"op": "get_folder_stats_batch", "arg": ["root0", "root1/sub0", ""]})
    ops.append({"op": "get_file_chunk_counts", "arg": "root2"})
    ops.append({"op": "set_file_acl", "args": [m0["file_path"], ["a@x.org", "b@x.org"]]})
    ops.append({"op": "get_chunks_by_range", "args": [m0["file_path"], 0, 0]})
    # (x) deletes change N and df used by the IDF
    ops.append({"op": "delete_by_file", "arg": corpus["metas"][3]["file_path"]})
    ops.append({"op": "delete_by_file", "arg": "nope"})
    ops.append({"op": "delete_by_folder", "arg": folders[2]})
    S(0, limit=10, sparse=True)
    S(1, limit=10, sparse=False)
    ops.append({"op": "delete_by_index_folder", "arg": "root1"})
    S(0, limit=10, sparse=True)
    S(4, limit=10, sparse=True, exclude_index_folders=["root0"])
    ops.append({"op": "info"})
    # re-ingest after deletes
    ops.append({"op": "store", "lo": 0, "hi": 60, "sparse": True})
    S(0, limit=10, sparse=True)
    ops.append({"op": "info"})
    return ops


def special_sparse(kind, corpus, qi, queries):
    """Resolve the symbolic sparse-query kinds used in ``scenario``."""
    if kind is True:
        return queries[qi][1]
    if kind is False:
        return None
    if kind == "empty":
        return ([], [])
    if kind == "absent":
        return ([2**31 - 5], [1.0])
    # find the rarest term (df == 1 -> 'single'; a few hits -> 'rare')
    df: dict[int, int] = {}
    for r, (idx, _) in enumerate(corpus["sparse"]):
        if 400 <= r < 450:
            continue
        for t in idx:
            df[t] = df.get(t, 0) + 1
    by = sorted(df.items(), key=lambda kv: (kv[1], kv[0]))
    if kind == "single":
        t = next(t for t, c in by if c == 1)
        return ([t], [1.0])
    if kind == "rare":
        ts = [t for t, c in by if 2 <= c <= 4][:3]
        return (ts, [1.0] * len(ts))
    raise ValueError(kind)


def build_inputs():
    corpus = _data.make_corpus(seed=20251018, n=N, dim=DIM)
    # (ii) tie case: rows 10/11 identical (dense + sparse), row 12 a zero dense vector
    corpus["dense"][11] = corpus["dense"][10]
    corpus["sparse"][11] = (list(corpus["sparse"][10][0]), list(corpus["sparse"][10][1]))
    corpus["dense"][12] = 0.0
    queries = _data.make_queries(seed=7, corpus=corpus, nq=11)
    q10 = corpus["dense"][10] / np.linalg.norm(corpus["dense"][10])
    queries[10] = (_data.bf16_round(q10.astype(np.float32)), (corpus["sparse"][10][0][:4], [1.0] * 4))
    return corpus, queries


def replay(store, ops, corpus, queries, meta_cls, row_of: dict):
    """Run ``ops`` against any VectorStoreService-shaped object.  ``row_of`` maps id -> a
    stable label ("<insertion row>" or "<row>#<generation>").  Returns the list of outputs."""
    outs = []
    gen: dict[int, int] = {}
    for op in ops:
        k = op["op"]
        if k == "store":
            lo, hi = op["lo"], op["hi"]
            chunks = [(corpus["texts"][r], corpus["dense"][r].astype(float).tolist(), meta_cls(**corpus["metas"][r]))
                      for r in range(lo, hi)]
            sv = [corpus["sparse"][r] for r in range(lo, hi)] if op["sparse"] else None
            kw = {"batch_size": op["batch_size"]} if "batch_size" in op else {}
            ids = store.store_chunks(chunks, sv, **kw)
            for r, pid in zip(range(lo, hi), ids):
                g = gen.get(r, 0)
                gen[r] = g + 1
                row_of[pid] = f"{r}" if g == 0 else f"{r}#{g}"
            outs.append(len(ids))
        elif k == "search":
            kw = dict(op["kw"])
            sq = special_sparse(kw.pop("sparse"), corpus, op["q"], queries)
            res = store.search(queries[op["q"]][0].astype(float).tolist(), sparse_query=sq, **kw)
            outs.append([[row_of[c.id], c.score, c.metadata.file_path, c.metadata.index_folder] for c in res])
        elif k == "info":
            info = store.get_collection_info()
            outs.append(info.get("points_count"))
        elif k in ("get_chunks_by_range", "find_by_source_url"):
            res = getattr(store, k)(*(op["args"] if "args" in op else [op["arg"]]))
            outs.append([[row_of[c.id], c.metadata.chunk_index, c.metadata.allowed_users] for c in res])
        elif k == "set_file_acl":
            store.set_file_acl(*op["args"])
            outs.append(None)
        elif k == "get_file_paths_by_index_folder":
            outs.append(sorted(store.get_file_paths_by_index_folder(op["arg"])))
        elif k in ("count_chunks_for_folder",):
            outs.append(list(store.count_chunks_for_folder(op["arg"])))
        elif k == "get_folder_stats_batch":
            outs.append({a: list(b) for a, b in store.get_folder_stats_batch(op["arg"]).items()})
        else:
            outs.append(getattr(store, k)(op["arg"]))
    return outs


def check_against_real_qdrant():
    """Replay the scenario through the reference over the REAL qdrant-client and compare with the committed
    golden file (generated over the oracle).  Any difference means the oracle's restatement of qdrant-client
    is wrong: fail loudly.  Returns the number of operations compared."""
    sys.path.insert(0, str(ROOT / "tests"))
    from _parity import assert_same_ranking
    corpus, queries = build_inputs()
    gold = json.loads((Path(__file__).resolve().parent / "voitta_cases.json").read_text())
    ref = load_reference_vector_store(DIM, real=True)
    store = ref.VectorStoreService()
    outs = replay(store, gold["ops"], corpus, queries, ref.ChunkMetadata, {})
    assert len(outs) == len(gold["outs"])
    for i, (op, got, want) in enumerate(zip(gold["ops"], outs, gold["outs"])):
        what = f"real qdrant-client vs oracle golden, op {i} {op}"
        if op["op"] == "search":
            assert_same_ranking(got, want, rel_tol=1e-5, abs_tol=2e-6, what=what)
        else:
            assert json.loads(json.dumps(got)) == want, what
    return len(outs)


def main():
    if real_qdrant_available():
        n = check_against_real_qdrant()
        print(f"qdrant-client is installed: {n} golden operations re-checked against it — the oracle is PINNED")
        return
    corpus, queries = build_inputs()
    ops = scenario(corpus, queries)
    ref = load_reference_vector_store(DIM)
    counter = iter(range(1, 10**9))
    real_uuid4 = uuid.uuid4
    uuid.uuid4 = lambda: uuid.UUID(int=(next(counter) * 0x9E3779B97F4A7C15) % (1 << 128))
    try:
        store = ref.VectorStoreService()
        outs = replay(store, ops, corpus, queries, ref.ChunkMetadata, {})
    finally:
        uuid.uuid4 = real_uuid4
    out_dir = Path(__file__).resolve().parent
    with open(out_dir / "voitta_cases.json", "w") as f:
        json.dump({"generated_by": "tests/golden/make_golden.py",
                   "reference": "voitta/services/vector_store.py (unmodified) over "
                                "oracle.LocalCollection standing in for qdrant-client",
                   "dim": DIM, "n": N, "ops": ops, "outs": outs}, f, indent=0)
    n_search = sum(1 for o in ops if o["op"] == "search")
    print(f"wrote {out_dir / 'voitta_cases.json'}: {len(ops)} ops ({n_search} searches)")


if __name__ == "__main__":
    main()
