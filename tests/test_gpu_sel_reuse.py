"""The row selection (dense_compact.cuh) keeps its copy of the rows that pass a batch-wide filter across batches while
the filter's content, the index's write generation and the segment plan stay the same (option sel_reuse, vb_api.cu
run_branches).  Every case runs each batch with sel_reuse = 1 and then with sel_reuse = 0 on the same index: the keys
must be identical, the kept copy must save exactly the three launches per selected segment, and the answer must
match the oracle.  After a write the kept copy would be stale, so each write case also checks the rows the write
adds or removes."""
import numpy as np
import pytest

import _data
from _parity import assert_same_ranking
from oracle import oracle_c

pytestmark = pytest.mark.gpu

N, DIM, LIMIT = 150_000, 128, 10
TS_MODIFIED, LO, HI = 2, 1420070400, 1767225600
# seg_first 2048, growth 8: segments [2048, 16384), [16384, 131072), [131072, N) take the selection at
# dense_compact_min_rows = 1024 (the first one is the direct segment)
SELECTED = 3
SAVED = 3 * SELECTED


def scope_filter(ids, lo=LO, hi=HI, words=4):
    bits = np.zeros(words, np.uint32)
    for s in ids:
        bits[s >> 5] |= np.uint32(1 << (s & 31))
    return (bits, TS_MODIFIED, lo, hi)


FA = scope_filter(range(0, 100, 2))
FB = scope_filter(range(1, 100, 2), 1450000000, 1767225600)


class World:
    """One index plus the host copy of its rows, for the oracle."""

    def __init__(self, seed=11, n=N):
        from voitta_rag_b200 import engine
        rng = np.random.RandomState(seed)
        cents = rng.randn(64, DIM).astype(np.float32)
        self.dense = _data.bf16_round(cents[rng.randint(0, 64, size=n)] + 0.6 * rng.randn(n, DIM).astype(np.float32))
        self.scope = rng.randint(0, 100, size=n).astype(np.uint32)
        self.modified = rng.randint(LO, HI, size=n).astype(np.int64)
        self.alive = np.ones(n, bool)
        self.rng = rng
        self.ix = engine.Index(DIM)
        self.ix.upsert(self.dense, None, self.scope, None, self.modified)
        self.ix.set_option("dense_compact", 70)
        self.ix.set_option("dense_compact_min_rows", 1024)

    def queries(self, B, seed):
        r = np.random.RandomState(seed)
        return _data.bf16_round(self.dense[r.randint(0, len(self.dense), size=B)] + 0.3 * r.randn(B, DIM).astype(np.float32))

    def upsert(self, dense, scope, modified):
        first = self.ix.upsert(dense, None, scope, None, modified)
        self.dense = np.concatenate([self.dense, dense])
        self.scope = np.concatenate([self.scope, scope])
        self.modified = np.concatenate([self.modified, modified])
        self.alive = np.concatenate([self.alive, np.ones(len(dense), bool)])
        return first

    def delete(self, rows):
        self.ix.delete_rows(np.asarray(rows, np.uint64))
        self.alive[np.asarray(rows, np.int64)] = False

    def passing(self, f):
        bits = np.asarray(f[0], np.uint32)
        sc = self.scope
        ok = np.zeros(len(sc), bool)
        inb = (sc >> 5) < len(bits)
        ok[inb] = ((bits[sc[inb] >> 5] >> (sc[inb] & 31)) & 1).astype(bool)
        return ok & (self.modified >= f[2]) & (self.modified <= f[3]) & self.alive

    def close(self):
        self.ix.close()


def search(ix, Q, filters, filter_of=None, reuse=1):
    from voitta_rag_b200 import engine
    ix.set_option("sel_reuse", reuse)
    fo = np.zeros(len(Q), np.int32) if filter_of is None else np.asarray(filter_of, np.int32)
    res = ix.search_batch(Q, None, [engine.Filter(*f) for f in filters], fo, limit=LIMIT, fusion="dense", branches=True)
    return res, ix.stats()


def same(a, b, what):
    for name in ("rows", "scores", "counts", "dense_rows", "dense_scores", "dense_counts"):
        assert np.array_equal(getattr(a, name), getattr(b, name)), f"{what}: {name} differs between sel_reuse 1 and 0"


def pair(w, Q, filters, filter_of=None, what=""):
    """The batch with the kept copy (when its key holds), then copied afresh: identical answers and selection stats.
    Returns (result, launches saved by sel_reuse = 1)."""
    r1, s1 = search(w.ix, Q, filters, filter_of, 1)
    r0, s0 = search(w.ix, Q, filters, filter_of, 0)
    same(r1, r0, what)
    for k in ("last_sel_rows", "last_sel_used", "last_dense_path", "last_big_rows"):
        assert s1[k] == s0[k], (what, k, s1[k], s0[k])
    return r1, s0["last_launches"] - s1["last_launches"]


def check_oracle(w, Q, res, f, what, n_check=24):
    cc = oracle_c.CorpusC(w.dense, None, w.scope, None, w.modified, alive=w.alive.astype(np.uint8))
    sub = np.arange(min(n_check, len(Q)))
    want = cc.search_batch(Q[sub], None, [f], np.zeros(len(sub), np.int32), limit=LIMIT, kprime=LIMIT, fusion=0)
    tol = 1e-3 if len(Q) > 256 else 2e-5                  # plain bf16 query (K2T) / bf16x2 query (resident K2)
    passing = w.passing(f)
    for j, i in enumerate(sub):
        got = res.branch(i, "dense")
        assert passing[[r for r, _ in got]].all(), f"{what} q{i}: a returned row fails the filter or is deleted"
        wd = [(int(want["dense_rows"][j, t]), float(want["dense_scores"][j, t])) for t in range(want["dense_counts"][j])]
        assert_same_ranking(got, wd, rel_tol=tol, abs_tol=tol, what=f"{what} q{i}")


@pytest.fixture(scope="module")
def world():
    w = World()
    yield w
    w.close()


@pytest.mark.parametrize("B", [320, 40])
def test_same_filter_on_many_batches_keeps_the_copy(world, B):
    """B = 320: K2T (query-tiled), B = 40: resident K2.  The first batch copies; every later one keeps the copy."""
    world.ix.set_option("sel_reuse", 0)
    search(world.ix, world.queries(B, 0), [FB])            # the scratch holds another filter's selection
    for step in range(4):
        Q = world.queries(B, 100 + step)
        res, saved = pair(world, Q, [FA], what=f"B={B} step {step}")
        assert world.ix.stats()["last_dense_path"] == 2
        assert world.ix.stats()["last_sel_used"] == 1
        assert saved == (0 if step == 0 else SAVED), (step, saved)
        if step in (0, 3):
            check_oracle(world, Q, res, FA, f"B={B} step {step}")


def test_alternating_filters_and_content_equal_copies(world):
    """A, B, A: each change of filter copies again.  A copy of A as a new object with trailing zero scope words keeps
    A's selection, alone and beside A in one batch (the two merge into one batch-wide filter)."""
    B = 320
    a_copy = (np.concatenate([FA[0].copy(), np.zeros(7, np.uint32)]), FA[1], FA[2], FA[3])
    search(world.ix, world.queries(B, 1), [FA], reuse=0)
    expected = [(FB, 0), (FA, 0), (FA, SAVED), (a_copy, SAVED)]
    for step, (f, want_saved) in enumerate(expected):
        Q = world.queries(B, 200 + step)
        res, saved = pair(world, Q, [f], what=f"step {step}")
        assert saved == want_saved, (step, saved)
    Q = world.queries(B, 300)
    res, saved = pair(world, Q, [FA, a_copy], np.arange(B) % 2, what="A beside its copy")
    assert saved == SAVED
    check_oracle(world, Q, res, FA, "A beside its copy")


WRITES = ["delete_top_row", "upsert_query_row", "move_row_out_of_filter", "merge_past_delta_max"]


@pytest.mark.parametrize("write", WRITES)
def test_writes_invalidate_the_kept_copy(write):
    """The same filter before and after a write: the write's rows must show up (or vanish) in the next batch."""
    w = World(seed=23)
    try:
        B = 320
        Q = w.queries(B, 7)
        search(w.ix, Q, [FA], reuse=0)
        before, saved = pair(w, Q, [FA], what="before")
        assert saved == SAVED
        top = int(before.branch(0, "dense")[0][0])
        if write == "delete_top_row":
            w.delete([top])
        elif write in ("upsert_query_row", "merge_past_delta_max"):
            if write == "merge_past_delta_max":
                w.ix.optimize()                           # an index over every row: the next append is a delta
                w.ix.set_option("delta_max", 64)
            n_new = 1 if write == "upsert_query_row" else 100
            rows = w.queries(n_new, 99)
            rows[0] = Q[0]
            sc = np.full(n_new, 2, np.uint32)             # scope 2 passes FA
            first = w.upsert(rows, sc, np.full(n_new, 1600000000, np.int64))
            if write == "merge_past_delta_max":
                assert w.ix.stats()["delta_rows"] == 0, "100 rows past delta_max = 64 merge on the upsert"
        else:   # a passing row's scope changes: delete + append with a scope FA drops
            w.delete([top])
            first = w.upsert(w.dense[top:top + 1].copy(), np.array([3], np.uint32), w.modified[top:top + 1].copy())
        after, saved = pair(w, Q, [FA], what=write)
        assert saved == 0, "a write must make the next batch copy again"
        got = [r for r, _ in after.branch(0, "dense")]
        if write == "delete_top_row":
            assert top not in got
        elif write == "move_row_out_of_filter":
            assert top not in got and first not in got
        else:
            assert got[0] == first, (write, got[:3], first)
        check_oracle(w, Q, after, FA, write)
        again, saved = pair(w, w.queries(B, 8), [FA], what=write + " then again")
        assert saved == SAVED
    finally:
        w.close()


def test_per_query_filters_between_two_same_filter_batches(world):
    """A batch of 40 distinct per-query filters (mask mode 3) uses no selection and leaves the kept copy valid."""
    B = 320
    search(world.ix, world.queries(B, 2), [FA], reuse=0)
    fl = [scope_filter(range(i, 100, 40)) for i in range(40)]
    fo = np.arange(B) % 40
    Q = world.queries(B, 400)
    r1, s1 = search(world.ix, Q, fl, fo, 1)
    assert s1["last_sel_used"] == 0
    r0, s0 = search(world.ix, Q, fl, fo, 0)
    same(r1, r0, "per-query filters")
    assert s1["last_launches"] == s0["last_launches"]
    # the scratch still holds FA's selection (the per-query batches did not touch it)
    res, saved = pair(world, world.queries(B, 401), [FA], what="after per-query filters")
    assert saved == SAVED
    check_oracle(world, world.queries(B, 401), res, FA, "after per-query filters")


def test_safe_mode_segments_then_normal_batch(world):
    """The safe mode (the schedule of an overflow rerun) cuts other segments: it copies its own, and the next normal
    batch copies its segments again."""
    B = 320
    search(world.ix, world.queries(B, 3), [FA], reuse=0)
    world.ix.set_option("safe_mode", 1)
    try:
        Q = world.queries(B, 500)
        res, saved = pair(world, Q, [FA], what="safe mode")
        assert saved == 0
        check_oracle(world, Q, res, FA, "safe mode")
    finally:
        world.ix.set_option("safe_mode", 0)
    Q = world.queries(B, 501)
    r1, s1 = search(world.ix, Q, [FA], reuse=1)
    r0, s0 = search(world.ix, Q, [FA], reuse=0)
    same(r1, r0, "normal after safe mode")
    assert s1["last_launches"] == s0["last_launches"], "the normal segments must be copied again"
    check_oracle(world, Q, r1, FA, "normal after safe mode")


def test_two_in_flight_stream_equals_one_at_a_time(world):
    """search_stream (two batches in flight) over A, A, B, B, A equals the same batches run one at a time."""
    B = 320
    plan = [FA, FA, FB, FB, FA]
    Qs = [world.queries(B, 600 + i) for i in range(len(plan))]
    from voitta_rag_b200 import engine
    fo = np.zeros(B, np.int32)
    world.ix.set_option("sel_reuse", 1)
    packed = [world.ix.pack(Q, None, [engine.Filter(*f)], fo, limit=LIMIT, fusion="dense", branches=True) for Q, f in zip(Qs, plan)]
    streamed = list(world.ix.search_stream(iter(packed)))
    for i, (Q, f) in enumerate(zip(Qs, plan)):
        one, _ = search(world.ix, Q, [f], reuse=0)
        same(streamed[i], one, f"stream batch {i}")


def test_two_shards_merged_and_staged_with_kept_copies():
    """Two row shards under one filter, each keeping its copy across batches, merged as the multi-GPU layer does
    (stage, run_local, run_fuse(2, gathered), fetch): equal to the single index."""
    import torch
    from voitta_rag_b200 import engine
    w = World(seed=31, n=80_000)
    n, B = 80_000, 320
    halves = [engine.Index(DIM, row_base=0), engine.Index(DIM, row_base=n // 2)]
    try:
        for r, hx in enumerate(halves):
            s = slice(r * n // 2, (r + 1) * n // 2)
            hx.upsert(w.dense[s], None, w.scope[s], None, w.modified[s])
            hx.set_option("dense_compact", 70)
            hx.set_option("dense_compact_min_rows", 1024)
        words = engine.Index.cand_block_words(B, LIMIT)
        dev = torch.device("cuda", 0)
        fo = np.zeros(B, np.int32)
        for step in range(3):
            Q = w.queries(B, 700 + step)
            want, _ = search(w.ix, Q, [FA], reuse=0)
            gathered = torch.zeros(2 * words, dtype=torch.int64, device=dev)
            launches, staged = [], []
            for r, hx in enumerate(halves):
                staged.append(hx.stage(Q, None, [engine.Filter(*FA)], fo, limit=LIMIT, kprime=LIMIT, fusion="dense",
                                       apply_idf=False, branches=True))
                hx.run_local(gathered[r * words:].data_ptr())
                launches.append(hx.stats()["last_launches"])
            torch.cuda.synchronize()
            halves[0].run_fuse(2, gathered.data_ptr())
            merged = halves[0].fetch(staged[0])
            for i in range(B):
                assert merged.branch(i, "dense") == want.branch(i, "dense"), f"step {step} q{i}"
                assert merged.hits(i) == want.hits(i)
            if step == 0:
                first = launches
            else:
                assert all(l < f for l, f in zip(launches, first)), (step, launches, first)
    finally:
        for hx in halves:
            hx.close()
        w.close()


@pytest.mark.parametrize("option", ["dense_compact", "seg_ratio", "dense_path", "k2_tiled"])
def test_option_changes_between_batches(option):
    """An option that changes the selection plan makes the next batch copy again.  dense_path = 1 (the fp32 scan) uses
    no selection and leaves the scratch as it was, so the batch after it, back on the tensor cores, keeps the copy."""
    w = World(seed=41)
    B = 320
    try:
        search(w.ix, w.queries(B, 0), [FA], reuse=0)
        _, saved = pair(w, w.queries(B, 1), [FA], what="before")
        assert saved == SAVED
        old = {"dense_compact": 70, "seg_ratio": 0, "dense_path": 0, "k2_tiled": 1}[option]
        new = {"dense_compact": 100, "seg_ratio": 4, "dense_path": 1, "k2_tiled": 0}[option]
        w.ix.set_option(option, new)
        Q = w.queries(B, 2)
        res, saved = pair(w, Q, [FA], what=f"{option}={new}")
        if option == "dense_path":
            assert w.ix.stats()["last_dense_path"] == 1 and w.ix.stats()["last_sel_used"] == 0
        else:
            assert saved == 0, f"{option}={new} must copy again"
        check_oracle(w, Q, res, FA, f"{option}={new}")
        w.ix.set_option(option, old)
        Q = w.queries(B, 3)
        res, saved = pair(w, Q, [FA], what=f"{option} back")
        assert saved == (SAVED if option == "dense_path" else 0)
        check_oracle(w, Q, res, FA, f"{option} back")
    finally:
        w.close()
