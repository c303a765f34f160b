"""ACL filtering on the B200: no row a caller may not see comes back on any scoring path.

The scope ids of rows carry their allowed_users set (vector_store._Collection); set_file_acl rewrites them on the
device with vb_set_scope.  Every returned row of every branch list is held to a numpy predicate over the raw
allowed_users lists, and the lists to the C oracle given the folded bits (sparse bit-equal, dense at each path's
tolerance).  The host side of the feature is tests/test_host_acl.py."""
import threading

import numpy as np
import pytest

import _acl_data as A
import _data
from _acl_oracle import AclOracleVectorStore
from _parity import assert_same_list, assert_same_ranking
from oracle import oracle_c

pytestmark = pytest.mark.gpu

T0, T1 = 1420070400, 1767225600
# K1 / K1F score with the fp32 query; the tensor-core kernels take a bf16 query (plain on K2T, which also serves batches
# with per-query filters; hi + lo on the resident K2), so they are held to the wider of the two
DENSE_TOL = {1: 2e-5, 3: 2e-5, 2: 1e-3}


@pytest.fixture(scope="module")
def world():
    """200k x 128 hybrid rows over 40 folders and 300 ACL sets, with delta rows (appended after the index build),
    deletes and rewritten scopes; the scope dictionary is the host layer's, reached through a VectorStoreService."""
    from voitta_rag_b200 import engine
    from voitta_rag_b200 import vector_store as VS
    rng = np.random.RandomState(2024)
    n, n_base, dim, n_folders = 200_000, 176_000, 128, 40
    cents = rng.randn(256, dim).astype(np.float32)
    dense = _data.bf16_round(cents[rng.randint(0, 256, size=n)] + 0.7 * rng.randn(n, dim).astype(np.float32))
    vocab = np.unique(rng.randint(1, 2**31 - 1, size=8000).astype(np.int64))[:4000]
    p = 1.0 / np.arange(1, len(vocab) + 1) ** 1.07
    p /= p.sum()
    picks = np.sort(rng.choice(len(vocab), size=(n, 10), p=p), axis=1)
    rows_terms = [np.unique(vocab[picks[r]]) for r in range(n)]
    indptr = np.zeros(n + 1, np.int64)
    np.cumsum([len(t) for t in rows_terms], out=indptr[1:])
    terms = np.concatenate(rows_terms).astype(np.uint32)
    vals = (0.5 + 1.5 * rng.rand(len(terms))).astype(np.float32)
    modified = rng.randint(T0, T1, size=n).astype(np.int64)
    acls = A.acl_choices(300, 7)
    folder = rng.randint(0, n_folders, size=n)
    acl_of = rng.randint(0, len(acls), size=n)
    folders = [f"root{k % 3}/folder{k:03d}" for k in range(n_folders)]

    ix = engine.Index(dim)
    name = "gpu_acl_world"
    VS._drop_collection(name)
    svc = VS.VectorStoreService(_index_factory=lambda: ix)
    svc.collection_name, svc.dimension = name, dim
    coll = svc._coll

    def sid(r):
        return coll.scope_id(folders[folder[r]], f"root{folder[r] % 3}", VS._acl_of(acls[acl_of[r]]))

    scope = np.fromiter((sid(r) for r in range(n)), np.uint32, n)
    ix.upsert(dense[:n_base], (indptr[:n_base + 1], terms[:indptr[n_base]], vals[:indptr[n_base]]), scope[:n_base], None,
              modified[:n_base])
    ix.optimize()
    ix.set_option("delta_max", 1 << 20)                  # the rest stays a delta, scored from the forward index
    ip2 = indptr[n_base:] - indptr[n_base]
    ix.upsert(dense[n_base:], (ip2, terms[indptr[n_base]:], vals[indptr[n_base]:]), scope[n_base:], None, modified[n_base:])
    assert ix.stats()["delta_rows"] == n - n_base
    dead = rng.choice(n, size=n // 50, replace=False)
    ix.delete_rows(dead)
    alive = np.ones(n, bool)
    alive[dead] = False
    # rewritten ACLs, in the base and in the delta, some of them on deleted rows
    moved = np.unique(np.concatenate([rng.choice(n_base, 1500, replace=False), n_base + rng.choice(n - n_base, 300, replace=False),
                                      dead[:50]]))
    acl_of[moved] = rng.randint(0, len(acls), size=len(moved))
    new_ids = np.fromiter((sid(r) for r in moved), np.uint32, len(moved))
    ix.set_scope(moved, new_ids)
    scope[moved] = new_ids
    cc = oracle_c.CorpusC(dense, (indptr, terms, vals), scope, None, modified, alive=alive.astype(np.uint8))
    qrows = rng.randint(0, n, size=1024)
    Q = _data.bf16_round(dense[qrows] + 0.4 * rng.randn(1024, dim).astype(np.float32))
    SP = [list(dict.fromkeys(rows_terms[r][:5].tolist() + [int(vocab[rng.randint(0, len(vocab))])])) for r in qrows]
    SP = [(t, [1.0] * len(t)) for t in SP]
    yield dict(engine=engine, ix=ix, svc=svc, cc=cc, acls=acls, acl_of=acl_of, folder=folder, folders=folders, alive=alive,
               modified=modified, scope=scope, Q=Q, SP=SP, n=n)
    VS._drop_collection(name)


def visible_rows(w, spec):
    """The predicate over the raw allowed_users lists (and the folder / date clauses), independent of the fold."""
    principals, kw = spec
    acl_ok = np.array([A.visible(a, principals) for a in w["acls"]])
    ok = w["alive"] & acl_ok[w["acl_of"]]
    if kw.get("include_folders"):
        fok = np.isin(np.arange(len(w["folders"])), [w["folders"].index(f) for f in kw["include_folders"]])
        ok &= fok[w["folder"]]
    if kw.get("date_start") is not None:
        ok &= (w["modified"] >= kw["date_start"]) & (w["modified"] <= kw["date_end"])
    return ok


def specs_for(w, count, seed):
    """`count` (principals, folder / date clause) pairs: every third one adds folders, every fifth a date range."""
    rng = np.random.RandomState(seed)
    out = []
    for k, p in enumerate(A.principal_lists(count, seed)):
        kw = {}
        if k % 3 == 1:
            kw["include_folders"] = sorted(rng.choice(w["folders"], size=rng.randint(5, 30), replace=False).tolist())
        if k % 5 == 2:
            lo = T0 + int(rng.randint(0, 150_000_000))
            kw.update(date_start=lo, date_end=lo + 150_000_000, date_field="modified")
        out.append((p, kw))
    return out


def run(w, B, specs, fo, options):
    eng, ix, svc = w["engine"], w["ix"], w["svc"]
    flts = [svc._build_filter(**kw, visible_to=p) for p, kw in specs]
    # a caller whose visibility passes every scope has no filter; the rest go to the library as they are
    fl_used, fo_used = [], np.full(B, -1, np.int32)
    for i in range(B):
        f = flts[fo[i]]
        if f is not None:
            fo_used[i] = len(fl_used)
            fl_used.append(f)
    for k, v in options.items():
        ix.set_option(k, v)
    try:
        got = ix.search_batch(w["Q"][:B], w["SP"][:B], fl_used or None, fo_used if fl_used else None, limit=20,
                              fusion="rrf", branches=True)
        st = ix.stats()
    finally:
        for k, v in (("dense_path", 0), ("k1f", 1), ("dense_compact", -1), ("dense_compact_min_rows", 1 << 18)):
            ix.set_option(k, v)
    return got, st, fl_used, fo_used


def check(w, got, B, specs, fo, fl_used, fo_used, path, what):
    vis = {}
    for i in range(B):
        k = int(fo[i])
        if k not in vis:
            vis[k] = visible_rows(w, specs[k])
        for br in ("dense", "sparse"):
            rows = [r for r, _ in got.branch(i, br)]
            assert len(set(rows)) == len(rows), f"{what} {br} q{i}: duplicate rows"
            assert vis[k][rows].all(), f"{what} {br} q{i}: a row the caller may not see came back"
        assert len(got.branch(i, "dense")) == min(60, int(vis[k].sum())), f"{what} q{i}: short list"
    sub = np.unique(np.linspace(0, B - 1, min(B, 24)).astype(int))
    tup = [(f.scope_bits, f.ts_field, f.ts_lo, f.ts_hi) for f in fl_used] or None
    want = w["cc"].search_batch(w["Q"][sub], [w["SP"][i] for i in sub], tup, fo_used[sub] if tup else None,
                                limit=20, kprime=60, fusion=2)
    tol = DENSE_TOL[path]
    for j, i in enumerate(sub):
        wd = [(int(want["dense_rows"][j, t]), float(want["dense_scores"][j, t])) for t in range(want["dense_counts"][j])]
        assert_same_ranking(got.branch(i, "dense"), wd, rel_tol=tol, abs_tol=tol, what=f"{what} dense q{i}")
        ws = [(int(want["sparse_rows"][j, t]), float(want["sparse_scores"][j, t])) for t in range(want["sparse_counts"][j])]
        assert_same_list(got.branch(i, "sparse"), ws, what=f"{what} sparse q{i}")


PATHS = {"K1F": ({"dense_path": 1, "k1f": 1}, 3), "K1": ({"dense_path": 1, "k1f": 0}, 1), "K2": ({"dense_path": 2}, 2),
         "K2-rowsel": ({"dense_path": 2, "dense_compact": 100, "dense_compact_min_rows": 1024}, 2)}


# K1F serves batches of at most 8 queries; K1 runs one pass per query, so B = 256 stands for the large batches; the row
# selection serves batch-wide filters only
CASES = [(path, mode, B) for path in PATHS for mode in ("per_query", "shared") for B in (1, 8, 256, 1024)
         if not (path == "K1F" and B > 8) and not (path == "K1" and B == 1024)
         and not (path == "K2-rowsel" and mode == "per_query")]


@pytest.mark.parametrize("path,mode,B", CASES)
def test_no_row_leaks_on_any_path(world, path, mode, B):
    w = world
    options, want_path = PATHS[path]
    if mode == "per_query":
        specs = specs_for(w, min(B, 64), seed=B)
        fo = (np.arange(B) % len(specs)).astype(np.int32)
    else:
        specs = [([A.USERS[3], A.GROUPS[1]], {})]
        fo = np.zeros(B, np.int32)
    got, st, fl_used, fo_used = run(w, B, specs, fo, options)
    assert st["last_dense_path"] == want_path, st
    if path == "K2-rowsel":
        assert st["last_sel_used"] == 1, st
    check(w, got, B, specs, fo, fl_used, fo_used, want_path, f"{path} {mode} B={B}")


def test_set_scope_errors_and_shards():
    """vb_set_scope: global rows on a shard, the errors it names a row in, and a two-shard merge equal to one index."""
    import torch
    from voitta_rag_b200 import engine
    rng = np.random.RandomState(5)
    n, dim, half = 40_000, 128, 20_000
    dense = _data.bf16_round(rng.randn(n, dim).astype(np.float32))
    scope = rng.randint(0, 60, size=n).astype(np.uint32)
    single = engine.Index(dim)
    shards = [engine.Index(dim, row_base=0), engine.Index(dim, row_base=half)]
    try:
        single.upsert(dense, None, scope)
        for hx, (lo, hi) in zip(shards, ((0, half), (half, n))):
            hx.upsert(dense[lo:hi], None, scope[lo:hi])
        for bad, msg in (([half - 1], str(half - 1)), ([n], str(n)), ([half + 5, half + 9, half + 5], str(half + 5))):
            with pytest.raises(engine.B200Error, match=msg):
                shards[1].set_scope(np.asarray(bad, np.uint64), np.zeros(len(bad), np.uint32))
        with pytest.raises(engine.B200Error, match=str(n)):
            single.set_scope([n], [0])
        with pytest.raises(engine.B200Error, match="twice"):
            single.set_scope([7, 3, 7], [1, 2, 3])
        single.set_scope(np.zeros(0, np.uint64), np.zeros(0, np.uint32))        # nothing to do
        single.delete_rows([11])
        shards[0].delete_rows([11])
        moved = rng.choice(n, 4000, replace=False)
        ids = rng.randint(60, 64, size=len(moved)).astype(np.uint32)              # scopes 60..63 only through the rewrite
        moved = np.append(moved, 11).astype(np.uint64)                            # a deleted row is accepted
        ids = np.append(ids, 62).astype(np.uint32)
        single.set_scope(moved, ids)
        for hx, (lo, hi) in zip(shards, ((0, half), (half, n))):
            m = (moved >= lo) & (moved < hi)
            hx.set_scope(moved[m], ids[m])                                         # global ids on both shards
        scope[moved.astype(np.int64)] = ids
        B, limit = 64, 20
        Q = _data.bf16_round(dense[rng.randint(0, n, size=B)] + 0.3 * rng.randn(B, dim).astype(np.float32))
        bits = np.zeros(2, np.uint32)
        bits[1] = np.uint32(0xF0000000)                                            # scopes 60..63
        gf = [engine.Filter(bits)]
        fo = np.zeros(B, np.int32)
        want = single.search_batch(Q, None, gf, fo, limit=limit, fusion="dense", branches=True)
        alive = np.ones(n, bool)
        alive[11] = False
        ok = (scope >= 60) & alive
        for i in range(B):
            assert ok[[r for r, _ in want.branch(i, "dense")]].all()
        words = engine.Index.cand_block_words(B, limit)
        gathered = torch.zeros(2 * words, dtype=torch.int64, device="cuda")
        for r, hx in enumerate(shards):
            hx.search_local(gathered[r * words:].data_ptr(), Q, None, gf, fo, limit=limit, kprime=limit, fusion="dense")
        torch.cuda.synchronize()
        merged = shards[0].merge_fuse(gathered.data_ptr(), 2, Q, None, limit=limit, kprime=limit, fusion="dense", branches=True)
        for i in range(B):
            assert merged.branch(i, "dense") == want.branch(i, "dense"), f"q{i}"
        assert any(r >= half for i in range(B) for r, _ in merged.branch(i, "dense"))
    finally:
        single.close()
        for hx in shards:
            hx.close()


# ---- the service ------------------------------------------------------------------------------------------------
DIM = 64


@pytest.fixture()
def service(monkeypatch):
    from voitta_rag_b200 import vector_store as VS
    name = "gpu_acl_service"
    monkeypatch.setenv("QDRANT_COLLECTION", name)
    monkeypatch.setenv("EMBEDDING_DIMENSION", str(DIM))
    VS._drop_collection(name)
    yield VS
    VS._drop_collection(name)


def fill(VS, store, n_files, seed):
    chunks, sparse = A.make_chunks(VS.ChunkMetadata, n_files, 10, DIM, 20, A.acl_choices(40, seed), seed)
    chunks = [(t, _data.bf16_round(np.asarray(e, np.float32)).tolist(), m) for t, e, m in chunks]   # what the device stores
    ids = store.store_chunks(chunks, sparse)
    return chunks, sparse, ids


def pairs(res):
    return [(c.id, c.score) for c in res]


@pytest.mark.parametrize("fusion", ["weighted", "rrf"])
def test_service_against_the_python_oracle(service, fusion):
    VS = service
    store = VS.VectorStoreService()
    store.fusion = fusion
    chunks, sparse, ids = fill(VS, store, 60, 3)
    ref = AclOracleVectorStore(DIM, fusion=fusion)
    ref.store_chunks(chunks, sparse, ids=ids)
    files = sorted({m.file_path for _, _, m in chunks})
    for fp, acl in ((files[0], [A.USERS[1]]), (files[1], []), (files[2], None), (files[3], [A.GROUPS[0], "x@y.org"])):
        store.set_file_acl(fp, acl)
        ref.set_file_acl(fp, acl)
    rng = np.random.RandomState(1)
    plist = A.principal_lists(8, 3)
    qs = [_data.bf16_round(rng.standard_normal(DIM).astype(np.float32)).tolist() for _ in plist]
    sqs = [(rng.choice(4000, 6, replace=False).tolist(), rng.uniform(0.5, 2, 6).tolist()) for _ in plist]
    for q, sq, p in zip(qs, sqs, plist):
        got = store.search_visible(q, 10, sparse_query=sq, visible_to=p)
        assert_same_ranking(pairs(got), pairs(ref.search(q, 10, sparse_query=sq, visible_to=p)), rel_tol=1e-4, abs_tol=1e-5)
        assert all(A.visible(c.metadata.allowed_users, p) for c in got)
    # batches may take a tensor-core path (bf16 query operand)
    batch = store.search_batch(qs, 10, sparse_queries=sqs, filters=[{"visible_to": p} for p in plist])
    for q, sq, p, got in zip(qs, sqs, plist, batch):
        assert_same_ranking(pairs(got), pairs(ref.search(q, 10, sparse_query=sq, visible_to=p)), rel_tol=1e-3, abs_tol=1e-3)
        assert all(A.visible(c.metadata.allowed_users, p) for c in got)
    shared = store.search_batch(qs, 10, sparse_queries=sqs, visible_to=plist[3])
    for q, sq, got in zip(qs, sqs, shared):
        assert_same_ranking(pairs(got), pairs(ref.search(q, 10, sparse_query=sq, visible_to=plist[3])), rel_tol=1e-3, abs_tol=1e-3)
        assert all(A.visible(c.metadata.allowed_users, plist[3]) for c in got)


def test_revocation_between_batches(service):
    """A batch under one shared visible_to keeps its row selection; set_file_acl then takes the user off files in its
    top results: the next batch drops those rows, copies the selection again and equals the oracle.  A batch staged
    before the write is refused."""
    VS = service
    from voitta_rag_b200 import engine
    store = VS.VectorStoreService()
    chunks, _, ids = fill(VS, store, 4000, 8)
    ix = store.client
    user = A.USERS[0]
    for fp in sorted({m.file_path for _, _, m in chunks})[::4]:     # a quarter of the files: the user alone may see them
        store.set_file_acl(fp, [user])
    rng = np.random.RandomState(2)
    Q = np.stack([np.asarray(chunks[i][1], np.float32) for i in rng.randint(0, len(chunks), 64)])
    Q = _data.bf16_round(Q + 0.05 * rng.randn(*Q.shape).astype(np.float32))
    ix.set_option("dense_path", 2)
    ix.set_option("dense_compact", 100)
    ix.set_option("dense_compact_min_rows", 1024)
    try:
        store.search_batch(Q, 20, visible_to=[user])
        before = store.search_batch(Q, 20, visible_to=[user])
        st = ix.stats()
        assert st["last_sel_used"] == 1 and st["last_dense_path"] == 2, st
        coll = store._coll
        revoked = {c.metadata.file_path for res in before for c in res[:5] if c.metadata.allowed_users == [user]}
        assert revoked, "no restricted file among the top results"
        flt = store._build_filter(visible_to=[user])
        staged = ix.stage(Q, None, [flt], np.zeros(len(Q), np.int32), limit=20, fusion="dense")
        for fp in sorted(revoked):
            store.set_file_acl(fp, ["someone-else@x.org"])
        with pytest.raises(engine.B200Error):
            ix.run_local()
        del staged
        after = store.search_batch(Q, 20, visible_to=[user])
        l1 = ix.stats()["last_launches"]
        assert all(c.metadata.file_path not in revoked for res in after for c in res)
        assert any(c.metadata.file_path in revoked for res in before for c in res)
        ix.set_option("sel_reuse", 0)
        fresh = store.search_batch(Q, 20, visible_to=[user])
        assert ix.stats()["last_launches"] == l1                  # the batch after the write copied the selection itself
        ix.set_option("sel_reuse", 1)
        assert [pairs(r) for r in after] == [pairs(r) for r in fresh]
        # oracle: the C oracle over the host copy of the rows, with the bits the host layer folds now
        rows = np.stack([np.asarray(c[1], np.float32) for c in chunks])
        cc = oracle_c.CorpusC(rows, None, ix_scope(coll), None, None)
        f = store._build_filter(visible_to=[user])
        want = cc.search_batch(Q, None, [(f.scope_bits, f.ts_field, f.ts_lo, f.ts_hi)], np.zeros(len(Q), np.int32),
                               limit=20, kprime=20, fusion=0)
        row_of = {pid: r for r, pid in enumerate(coll.ids)}
        for i, res in enumerate(after):
            wd = [(int(want["rows"][i, t]), float(want["scores"][i, t])) for t in range(want["counts"][i])]
            assert_same_ranking([(row_of[c.id], c.score) for c in res], wd, rel_tol=2e-5, abs_tol=2e-5, what=f"q{i}")
    finally:
        for k, v in (("dense_path", 0), ("dense_compact", -1), ("dense_compact_min_rows", 1 << 18), ("sel_reuse", 1)):
            ix.set_option(k, v)


def ix_scope(coll):
    """The scope id the host layer gives each row now (what vb_set_scope wrote on the device)."""
    from voitta_rag_b200 import vector_store as VS
    return np.fromiter((coll.scopes[(p["folder_path"], p["index_folder"])] if p.get("allowed_users") is None else
                        coll.scopes[(p["folder_path"], p["index_folder"], coll.acl_ids[VS._acl_of(p["allowed_users"])])]
                        for p in coll.payload), np.uint32, len(coll.payload))


def test_persistence_and_concurrency(service, tmp_path):
    VS = service
    store = VS.VectorStoreService()
    chunks, sparse, _ = fill(VS, store, 400, 12)
    files = sorted({m.file_path for _, _, m in chunks})
    for k, fp in enumerate(files[:40]):
        store.set_file_acl(fp, [A.USERS[k % 5]] if k % 3 else [])
    plist = A.principal_lists(16, 12)
    rng = np.random.RandomState(4)
    qs = [_data.bf16_round(rng.standard_normal(DIM).astype(np.float32)).tolist() for _ in plist]
    sqs = [(rng.choice(4000, 6, replace=False).tolist(), rng.uniform(0.5, 2, 6).tolist()) for _ in plist]
    single = [pairs(store.search_visible(q, 10, sparse_query=sq, visible_to=p)) for q, sq, p in zip(qs, sqs, plist)]
    # 16 threads, one caller identity each, coalesced into shared device batches
    out = [None] * len(plist)
    barrier = threading.Barrier(len(plist))

    def worker(k):
        barrier.wait()
        for _ in range(5):
            out[k] = pairs(store.search_visible(qs[k], 10, sparse_query=sqs[k], visible_to=plist[k]))

    th = [threading.Thread(target=worker, args=(k,)) for k in range(len(plist))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    for k in range(len(plist)):
        assert_same_ranking(out[k], single[k], rel_tol=1e-3, abs_tol=1e-3, what=f"thread {k}")
    # snapshot after the ACL writes (the device file carries the rewritten scope ids), restored into a new index
    store.save_snapshot(str(tmp_path))
    VS._drop_collection(store.collection_name)
    fresh = VS.VectorStoreService()
    fresh.load_snapshot(str(tmp_path))
    again = [pairs(fresh.search_visible(q, 10, sparse_query=sq, visible_to=p)) for q, sq, p in zip(qs, sqs, plist)]
    for k in range(len(plist)):
        # the restored index scores every row from a fresh inverted index: same rows, sums possibly in another order
        assert [r for r, _ in again[k]] == [r for r, _ in single[k]], f"restored q{k}"
        assert_same_ranking(again[k], single[k], rel_tol=1e-6, abs_tol=1e-7, what=f"restored q{k}")
