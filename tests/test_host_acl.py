"""ACL filtering through the host layer on a CPU box (VectorStoreService over the C-oracle test double): the folded
scope bitsets against a brute-force evaluation of every row's payload, the scope dictionary of ACL-free collections,
set_file_acl and its rollback, the argument errors, snapshots at versions 2 and 3, and search_visible against the
Python oracle.  The GPU side is tests/test_gpu_acl.py."""
import json

import numpy as np
import pytest

import _acl_data as A
from _acl_oracle import AclOracleVectorStore, ScopedFakeIndex
from _fake_index import FakeIndex
from _parity import assert_same_ranking
from oracle import oracle as O
from voitta_rag_b200 import engine
from voitta_rag_b200 import vector_store as VS

DIM = 16
NAME = "host_acl_test"


@pytest.fixture()
def store(monkeypatch):
    monkeypatch.setenv("QDRANT_COLLECTION", NAME)
    monkeypatch.setenv("EMBEDDING_DIMENSION", str(DIM))
    VS._drop_collection(NAME)
    s = VS.VectorStoreService(_index_factory=lambda: ScopedFakeIndex(DIM))
    yield s
    VS._drop_collection(NAME)


def fill(store, n_files=120, n_folders=9, n_acls=30, seed=0, acls=None):
    chunks, sparse = A.make_chunks(VS.ChunkMetadata, n_files, 3, DIM, n_folders,
                                   acls if acls is not None else A.acl_choices(n_acls, seed), seed)
    store.store_chunks(chunks, sparse)
    return sorted({m.folder_path for _, _, m in chunks})


def row_passes(f, ix: FakeIndex) -> np.ndarray:
    """What K0 computes for filter f over the index's columns (live rows only)."""
    ok = ix.alive.astype(bool).copy()
    if f is None:
        return ok
    if f.scope_bits is not None:
        sid = ix.scope.astype(np.int64)
        words = np.asarray(f.scope_bits, np.uint32)
        in_range = (sid >> 5) < len(words)
        bit = np.zeros(len(sid), bool)
        bit[in_range] = (words[sid[in_range] >> 5] >> (sid[in_range] & 31).astype(np.uint32)) & 1 == 1
        ok &= bit
    if f.ts_field != engine.TS_NONE:
        t = ix.created if f.ts_field == engine.TS_CREATED else ix.modified
        ok &= (t != engine.TS_MISSING) & (t >= f.ts_lo) & (t <= f.ts_hi)
    return ok


def brute(coll, kw, principals) -> np.ndarray:
    """Each row's payload through the Python oracle's filter, plus the ACL predicate stated in _acl_data."""
    flt = O.build_filter(**{k: v for k, v in kw.items() if k != "scope_key"})
    out = np.zeros(len(coll.payload), bool)
    for r, p in enumerate(coll.payload):
        if p is None:
            continue
        out[r] = O.check_filter(flt, p) and (principals is None or A.visible(p.get("allowed_users"), principals))
    return out


def same_filter(a, b):
    if a is None or b is None:
        return a is None and b is None
    return ((a.scope_bits is None) == (b.scope_bits is None) and (a.scope_bits is None or np.array_equal(a.scope_bits, b.scope_bits))
            and (a.ts_field, a.ts_lo, a.ts_hi) == (b.ts_field, b.ts_lo, b.ts_hi))


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_fold_equals_brute_force_per_row(store, seed):
    folders = fill(store, seed=seed)
    coll = store._coll
    # deletes and ACL changes after ingest, so that rows move between scopes and some scopes lose every row
    files = sorted(coll.by_file)
    store.delete_by_file(files[3])
    store.set_file_acl(files[5], [A.USERS[2], A.GROUPS[3]])
    store.set_file_acl(files[6], [])
    store.set_file_acl(files[7], None)
    oracle_ptr = A.principal_lists(14, seed) + [None]
    for kw in A.filter_specs(folders, 14, seed):
        for p in oracle_ptr:
            f = store._build_filter(**kw, visible_to=p)
            got = row_passes(f, coll.index)
            want = brute(coll, kw, p)
            assert np.array_equal(got, want), (kw, p, np.flatnonzero(got != want)[:10])


def test_acl_free_collection_keeps_pair_scopes_and_bits(store):
    folders = fill(store, acls=[None])
    coll = store._coll
    # the scope dictionary of the parent layout: one (folder_path, index_folder) pair per distinct pair, in order of
    # first appearance
    want = {}
    for p in coll.payload:
        want.setdefault((p["folder_path"], p["index_folder"]), len(want))
    assert coll.scope_list == list(want) and coll.acl_list == []
    assert [want[(p["folder_path"], p["index_folder"])] for p in coll.payload] == coll.index.scope.tolist()
    for kw in A.filter_specs(folders, 12, 5):
        base = store._build_filter(**kw)
        for p in A.principal_lists(6, 5):
            assert same_filter(store._build_filter(**kw, visible_to=p), base), (kw, p)


def test_visible_to_that_passes_everything_is_dropped(store):
    acls = [[A.USERS[i], A.GROUPS[i % 3]] for i in range(10)] + [None]
    folders = fill(store, acls=acls)
    everyone = A.USERS + A.GROUPS
    assert any(len(k) == 3 for k in store._coll.scope_list)
    for kw in A.filter_specs(folders, 10, 7):
        assert same_filter(store._build_filter(**kw, visible_to=everyone), store._build_filter(**kw)), kw
    assert store._build_filter(visible_to=everyone) is None
    # equal visibility, equal filter content: the library merges them into one mask
    a = store._build_filter(visible_to=[A.USERS[1]])
    b = store._build_filter(visible_to=[A.USERS[1], "unknown@x.org"])
    assert same_filter(a, b) and a is not None


def test_set_file_acl_moves_rows_and_rolls_back_when_the_device_call_fails(store):
    fill(store, acls=[None])
    coll = store._coll
    fp = sorted(coll.by_file)[0]
    rows = sorted(coll.by_file[fp])
    store.set_file_acl(fp, ["a@x.org", "b@x.org"])
    assert all(coll.payload[r]["allowed_users"] == ["a@x.org", "b@x.org"] for r in rows)
    sid = coll.index.scope[rows]
    assert all(len(coll.scope_list[s]) == 3 and coll.acl_list[coll.scope_list[s][2]] == {"a@x.org", "b@x.org"} for s in sid)
    assert [c.metadata.allowed_users for c in store.get_chunks_by_range(fp, 0, 10)] == [["a@x.org", "b@x.org"]] * len(rows)

    scope_before = coll.index.scope.copy()

    def boom(rows, scope_id):
        raise engine.B200Error("device write failed")

    coll.index.set_scope = boom
    with pytest.raises(engine.B200Error):
        store.set_file_acl(fp, ["c@x.org"])
    assert all(coll.payload[r]["allowed_users"] == ["a@x.org", "b@x.org"] for r in rows)
    assert np.array_equal(coll.index.scope, scope_before)
    # the host view still matches the device view: c@x.org sees none of the file, a@x.org all of it
    del coll.index.set_scope
    assert not row_passes(store._build_filter(visible_to=["c@x.org"]), coll.index)[rows].any()
    assert row_passes(store._build_filter(visible_to=["a@x.org"]), coll.index)[rows].all()
    store.set_file_acl("no/such/file", ["x"])                  # no rows: nothing to do


def test_scope_key_cache_with_different_principals(store):
    folders = fill(store, seed=3)
    coll = store._coll
    kw = {"include_folders": folders[:5], "scope_key": ("user", "project", 1)}
    first = store._build_filter(**kw)
    cached = coll.bits_cache[kw["scope_key"]][1].copy()
    for p in A.principal_lists(10, 3):
        f = store._build_filter(**kw, visible_to=p)
        assert np.array_equal(row_passes(f, coll.index), brute(coll, kw, p)), p
        assert np.array_equal(coll.bits_cache[kw["scope_key"]][1], cached)      # the folder fold is never narrowed in place
    assert same_filter(store._build_filter(**kw), first)
    # a new ACL scope invalidates the cached fold (scope_version), and the next call folds again
    store.set_file_acl(sorted(coll.by_file)[0], ["brand-new@x.org"])
    f = store._build_filter(**kw, visible_to=["brand-new@x.org"])
    assert np.array_equal(row_passes(f, coll.index), brute(coll, kw, ["brand-new@x.org"]))


def test_type_errors(store):
    fill(store, n_files=10)
    fp = sorted(store._coll.by_file)[0]
    q = [0.1] * DIM
    for bad in ("alice@x.org", b"alice", ["a@x.org", 3], [None]):
        with pytest.raises(TypeError):
            store._build_filter(visible_to=bad)
        with pytest.raises(TypeError):
            store.search_visible(q, visible_to=bad)
        with pytest.raises(TypeError):
            store.search_batch([q], visible_to=bad)
        with pytest.raises(TypeError):
            store.search_batch([q], filters=[{"visible_to": bad}])
        with pytest.raises(TypeError):
            store.set_file_acl(fp, bad)
    m = VS.ChunkMetadata("a/f", "a", "a", "f", 0, 1, 0, 1, "t", allowed_users="alice@x.org")
    n = store.get_collection_info()["points_count"]
    with pytest.raises(TypeError):
        store.store_chunks([("t", q, m)])
    assert store.get_collection_info()["points_count"] == n
    with pytest.raises(ValueError):
        store.search_batch([q], filters=[None], visible_to=["a@x.org"])
    with pytest.raises(TypeError):
        store.search_visible(q)                                   # the identity is a required keyword


def test_snapshot_versions_2_and_3(store, tmp_path):
    fill(store, acls=[None])
    coll = store._coll
    d2, d3 = tmp_path / "v2", tmp_path / "v3"
    store.save_snapshot(str(d2))
    head = json.loads((d2 / f"{NAME}.host.json").read_text())
    assert head["version"] == 2 and head["acl_list"] == []
    fp = sorted(coll.by_file)[0]
    store.set_file_acl(fp, ["b@x.org", "a@x.org"])
    store.set_file_acl(sorted(coll.by_file)[1], [])
    store.save_snapshot(str(d3))
    head = json.loads((d3 / f"{NAME}.host.json").read_text())
    assert head["version"] == 3 and sorted(map(tuple, head["acl_list"])) == [(), ("a@x.org", "b@x.org")]
    folders = sorted({p["folder_path"] for p in coll.payload})
    specs = A.filter_specs(folders, 6, 11)
    plist = A.principal_lists(6, 11) + [None]
    want = {(i, j): row_passes(store._build_filter(**kw, visible_to=p), coll.index) for i, kw in enumerate(specs) for j, p in enumerate(plist)}
    for d, ver in ((d2, 2), (d3, 3)):
        VS._drop_collection(NAME)
        fresh = VS.VectorStoreService(_index_factory=lambda: ScopedFakeIndex(DIM))
        fresh.load_snapshot(str(d), _index_loader=ScopedFakeIndex.load)
        c = fresh._coll
        if ver == 2:
            assert c.acl_list == [] and all(len(k) == 2 for k in c.scope_list)
            assert all(fresh._build_filter(visible_to=p) is None for p in plist)
        else:
            assert c.scope_list == coll.scope_list and c.acl_list == coll.acl_list
            for (i, j), w in want.items():
                assert np.array_equal(row_passes(fresh._build_filter(**specs[i], visible_to=plist[j]), c.index), w)
            # and it keeps taking ACL writes after the restore
            fresh.set_file_acl(fp, None)
            assert row_passes(fresh._build_filter(visible_to=[]), c.index)[sorted(c.by_file[fp])].all()


def test_scope_list_replaced_as_bench_does(store):
    fill(store, acls=[None, ["a@x.org"]])
    coll = store._coll
    # bench.py e2e_api: names every synthetic scope id with a folder pair and bumps scope_version by hand
    n_scopes = 64
    coll.scope_list = [(f"root/folder{s:05d}", "root") for s in range(n_scopes)]
    coll.scopes = {k: i for i, k in enumerate(coll.scope_list)}
    coll.scope_version += 1
    kw = {"include_folders": [coll.scope_list[s][0] for s in range(0, n_scopes, 3)], "scope_key": ("bench", 1)}
    base = store._build_filter(**kw)
    assert base.scope_bits.size == 2
    assert same_filter(store._build_filter(**kw, visible_to=["someone"]), base)
    assert store._build_filter(visible_to=[]) is None


@pytest.mark.parametrize("fusion", ["weighted", "rrf"])
def test_search_visible_and_search_batch_equal_the_oracle(store, fusion):
    chunks, sparse = A.make_chunks(VS.ChunkMetadata, 80, 3, DIM, 7, A.acl_choices(20, 4), 4)
    store.fusion = fusion
    ids = store.store_chunks(chunks, sparse)
    ref = AclOracleVectorStore(DIM, fusion=fusion)
    ref.store_chunks(chunks, sparse, ids=ids)
    files = sorted({m.file_path for _, _, m in chunks})
    for fp, acl in ((files[0], ["u1@x.org"]), (files[1], []), (files[2], None)):
        store.set_file_acl(fp, acl)
        ref.set_file_acl(fp, acl)
    rng = np.random.RandomState(9)
    folders = sorted({m.folder_path for _, _, m in chunks})
    plist = A.principal_lists(8, 4)
    specs = A.filter_specs(folders, len(plist), 4)
    qs = [rng.standard_normal(DIM).astype(np.float32).tolist() for _ in plist]
    sqs = [(rng.choice(4000, 6, replace=False).tolist(), rng.uniform(0.5, 2, 6).tolist()) for _ in plist]
    per_query = []
    for q, sq, p, kw in zip(qs, sqs, plist, specs):
        got = store.search_visible(q, 10, sparse_query=sq, visible_to=p, **kw)
        want = ref.search(q, 10, sparse_query=sq, visible_to=p, **kw)
        assert_same_ranking([(c.id, c.score) for c in got], [(c.id, c.score) for c in want], rel_tol=1e-5, abs_tol=2e-6)
        assert all(A.visible(c.metadata.allowed_users, p) for c in got)
        per_query.append([(c.id, c.score) for c in got])
    # one batch, one filter per query (visible_to in the dicts), and one batch under a shared visible_to
    batch = store.search_batch(qs, 10, sparse_queries=sqs, filters=[dict(kw, visible_to=p) for p, kw in zip(plist, specs)])
    for got, want in zip(batch, per_query):
        assert [(c.id, c.score) for c in got] == want
    shared = store.search_batch(qs, 10, sparse_queries=sqs, visible_to=plist[3])
    for q, sq, got in zip(qs, sqs, shared):
        want = ref.search(q, 10, sparse_query=sq, visible_to=plist[3])
        assert_same_ranking([(c.id, c.score) for c in got], [(c.id, c.score) for c in want], rel_tol=1e-5, abs_tol=2e-6)


def test_index_without_set_scope_fails_closed(store, tmp_path):
    """An index that cannot rewrite scope ids (the plain test double has no set_scope): set_file_acl updates the payloads
    as the reference does, searches without visible_to are unchanged, and visible_to is refused from then on, also
    after a snapshot round trip, instead of filtering by the rows' old scope ids."""
    VS._drop_collection(NAME)
    plain = VS.VectorStoreService(_index_factory=lambda: FakeIndex(DIM))
    fill(plain, acls=[None, ["a@x.org"]])
    coll = plain._coll
    assert plain._build_filter(visible_to=["a@x.org"]) is None       # no ACL changed yet: enforceable
    scope_before = coll.index.scope.copy()
    q = [0.1] * DIM
    want = [(c.id, c.score) for c in plain.search(q, 10)]
    fp = sorted(coll.by_file)[0]
    plain.set_file_acl(fp, ["b@x.org"])
    assert all(coll.payload[r]["allowed_users"] == ["b@x.org"] for r in coll.by_file[fp])
    assert np.array_equal(coll.index.scope, scope_before)
    assert [(c.id, c.score) for c in plain.search(q, 10)] == want
    for call in (lambda: plain.search_visible(q, visible_to=["b@x.org"]), lambda: plain._build_filter(visible_to=[]),
                 lambda: plain.search_batch([q], visible_to=["a@x.org"])):
        with pytest.raises(RuntimeError, match="cannot be enforced"):
            call()
    plain.save_snapshot(str(tmp_path))
    VS._drop_collection(NAME)
    fresh = VS.VectorStoreService(_index_factory=lambda: FakeIndex(DIM))
    fresh.load_snapshot(str(tmp_path), _index_loader=FakeIndex.load)
    with pytest.raises(RuntimeError, match="cannot be enforced"):
        fresh.search_visible(q, visible_to=["b@x.org"])
