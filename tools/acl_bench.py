"""Cost of ACL filtering on the cfg4 shard (12.5M x 768, hybrid RRF, top-100, batch 1024; bench.py's build_shard /
make_batches, whose filter is a folder scope set plus a date range over 4096 synthetic scopes).

Each of the 4096 scopes is split into k ACL variants (k = 1, 4, 32: up to 131k scope ids): the scope column is
rewritten with vb_set_scope (row r goes to variant hash(r) % k) and the host layer's scope dictionary names every
(folder, index folder, acl id).  Lines:

  none         bench.py's filter, no visible_to (compared bit for bit with the other builds given by --variant)
  k1           visible_to on an ACL-free dictionary: the clause drops out, the answers equal line none
  shared4/32   one visible_to for the whole batch (batch-wide filter: row selection reachable)
  distinct32   1024 distinct principal lists, one per query (1024 filters of 131k scope bits each)
  acl_write    set_file_acl of a 1000-chunk file (vb_set_scope of 1000 rows) and the batch after it
  fold         host fold per search_visible call at k = 32 (folder bits cached by scope_key, ACL part per call)

Every line is warmed, then timed for at least --min-seconds (search_packed: staging + H2D + kernels + D2H + decode)
with the profile option on for the phase times.  Each library build runs in its own child process (VB200_LIB); the
parent alternates the builds on line none --repeats times to show the spread and reads the card's name, power limit
and SM clock before and after.

    python tools/acl_bench.py --variant parent=/path/to/parent/libvoitta_b200.so,/path/to/parent/tree --out /tmp/acl_bench.json

A variant is NAME=LIB or NAME=LIB,TREE: with TREE its child imports the package and bench.py of that source tree (a
build from before vb_set_scope cannot be bound by this tree's engine.py).
"""
from __future__ import annotations

import sys

sys.dont_write_bytecode = True                      # the tree may be read-only

import argparse
import hashlib
import json
import os
import subprocess
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, os.environ.get("ACL_BENCH_TREE") or str(ROOT))

N_BASE_SCOPES = 4096


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else f"nvidia-smi failed: {r.stderr.strip()}"


# ---------------------------------------------------------------------------------------------- child: one library
def child():
    import torch
    import bench
    from voitta_rag_b200 import engine, synth
    from voitta_rag_b200 import vector_store as VS
    cfg = bench.WORKLOADS["cfg4"]
    device = torch.device("cuda", 0)
    ix, keep, (lo, hi), _ = bench.build_shard(cfg, 0, 1, device, torch, synth, engine)
    batches, flt_a = bench.make_batches(cfg, keep, 1, synth, engine, torch)
    batches = batches[:4]
    B, limit, n = cfg["batch"], cfg["limit"], hi - lo
    has_acl = hasattr(ix, "set_scope")
    base_scope = None

    def digest(res):
        h = hashlib.sha1()
        for a in (res.rows, res.scores, res.counts):
            h.update(np.ascontiguousarray(a).tobytes())
        return h.hexdigest()

    def timed(packs, min_s):
        for p in packs:
            ix.search_packed(p)
        digests = [digest(ix.search_packed(p)) for p in packs]
        ix.set_option("profile", 1)
        mask, dev_ms, steps, h2d, sel = 0.0, 0.0, 0, 0, 0
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        while True:
            ix.search_packed(packs[steps % len(packs)])
            st = ix.stats()
            mask += st["last_mask_ms"]
            dev_ms += st["last_search_ms"]
            h2d, sel = int(st["last_h2d_bytes"]), int(st["last_sel_used"])
            steps += 1
            el = time.perf_counter() - t0
            if el >= min_s and steps >= 2 * len(packs):
                break
        ix.set_option("profile", 0)
        return {"steps": steps, "step_ms": 1e3 * el / steps, "device_ms": dev_ms / steps, "mask_ms": mask / steps,
                "last_h2d_bytes": h2d, "last_sel_used": sel, "dense_path": int(ix.stats()["last_dense_path"]), "digests": digests}

    # the host layer over this shard: its scope dictionary names the synthetic scope ids
    os.environ["EMBEDDING_DIMENSION"] = str(cfg["dim"])
    os.environ["QDRANT_COLLECTION"] = "acl_bench"
    VS._drop_collection("acl_bench")
    svc = VS.VectorStoreService(_index_factory=lambda: ix)
    coll = svc._coll
    bits_a, _, ts_lo, ts_hi = flt_a
    folders = [f"root/folder{s:05d}" for s in range(N_BASE_SCOPES)]
    inc = [folders[s] for s in range(N_BASE_SCOPES) if s >> 5 < len(bits_a) and (int(bits_a[s >> 5]) >> (s & 31)) & 1]
    kw = {"include_folders": inc, "date_start": int(ts_lo), "date_end": int(ts_hi), "date_field": "modified"}

    def acl_split(k):
        """Scope s, variant j -> id s * k + j; row r takes variant hash(r) % k (the device column is rewritten)."""
        nonlocal base_scope
        if base_scope is None:
            parts = []
            for blk in range(lo // bench.BLOCK_ROWS, (hi + bench.BLOCK_ROWS - 1) // bench.BLOCK_ROWS):
                b_lo, b_hi = blk * bench.BLOCK_ROWS, min(cfg["n"], (blk + 1) * bench.BLOCK_ROWS)
                sc, _, _ = synth.columns(b_hi - b_lo, blk, device)
                parts.append(sc.cpu().numpy().astype(np.uint32)[max(lo, b_lo) - b_lo:min(hi, b_hi) - b_lo])
            base_scope = np.concatenate(parts)
        rows = np.arange(lo, hi, dtype=np.uint64)
        variant = ((rows * np.uint64(2654435761)) >> np.uint64(7)) % np.uint64(k)
        ids = (base_scope.astype(np.uint64) * np.uint64(k) + variant).astype(np.uint32)
        step = 2_000_000
        for a in range(0, n, step):
            ix.set_scope(rows[a:a + step], ids[a:a + step])
        coll.acl_list = [frozenset({f"user{j}@x.org", f"group{j % 4}"}) for j in range(k)] if k > 1 else []
        coll.acl_ids = {a: j for j, a in enumerate(coll.acl_list)}
        coll.scope_list = [(f, "root", j) for f in folders for j in range(k)] if k > 1 else [(f, "root") for f in folders]
        coll.scopes = {key: i for i, key in enumerate(coll.scope_list)}
        coll.scope_version += 1

    def packs_for(filters, fo):
        gf = [f for f in filters]
        return [ix.pack(q, sp, gf, fo, limit=limit, fusion="rrf") for q, sp in batches]

    def run_line(name, min_s):
        if name == "none":
            return timed(packs_for([engine.Filter(*flt_a)], np.zeros(B, np.int32)), min_s)
        if not has_acl:
            return {"skipped": "this build has no vb_set_scope"}
        if name == "k1":
            acl_split(1)
            f = svc._build_filter(**kw, scope_key=("bench", 1), visible_to=["user1@x.org"])
            return timed(packs_for([f], np.zeros(B, np.int32)), min_s)
        if name.startswith("shared"):
            k = int(name[6:])
            acl_split(k)
            f = svc._build_filter(**kw, scope_key=("bench", k), visible_to=["user1@x.org", "group2"])
            out = timed(packs_for([f], np.zeros(B, np.int32)), min_s)
            out.update(n_scopes=len(coll.scope_list), scope_words=int(f.scope_bits.size))
            return out
        if name == "distinct32":
            acl_split(32)
            rng = np.random.RandomState(32)
            plist = [[f"user{u}@x.org" for u in rng.choice(32, size=3, replace=False)] + [f"group{i % 4}"] for i in range(B)]
            t0 = time.perf_counter()
            fl = [svc._build_filter(**kw, scope_key=("bench", 32), visible_to=p) for p in plist]
            t1 = time.perf_counter()
            p0 = ix.pack(batches[0][0], batches[0][1], fl, np.arange(B, dtype=np.int32), limit=limit, fusion="rrf")
            t2 = time.perf_counter()
            out = timed(packs_for(fl, np.arange(B, dtype=np.int32)), min_s)
            distinct = len({f.scope_bits.tobytes() for f in fl})
            out.update(distinct_filters=distinct, scope_words=int(fl[0].scope_bits.size),
                       staged_scope_bytes=int(sum(f.scope_bits.nbytes for f in fl)),
                       host_fold_ms_batch=1e3 * (t1 - t0), host_pack_ms_batch=1e3 * (t2 - t1))
            del p0
            return out
        if name == "acl_write":
            acl_split(32)
            f = svc._build_filter(**kw, scope_key=("bench", 32), visible_to=["user1@x.org", "group2"])
            ps = packs_for([f], np.zeros(B, np.int32))
            steady = timed(ps, min_s)
            rng = np.random.RandomState(1000)
            lat, after = [], []
            for rep in range(5):
                rows = np.sort(rng.choice(n, 1000, replace=False)).astype(np.uint64) + np.uint64(lo)
                ids = rng.randint(0, len(coll.scope_list), size=1000).astype(np.uint32)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                ix.set_scope(rows, ids)
                lat.append(1e3 * (time.perf_counter() - t0))
                t0 = time.perf_counter()
                ix.search_packed(ps[rep % len(ps)])
                after.append(1e3 * (time.perf_counter() - t0))
            return {"set_scope_1000_rows_ms": lat, "first_batch_after_ms": after, "steady_step_ms": steady["step_ms"],
                    "steady_sel_used": steady["last_sel_used"]}
        if name == "fold":
            acl_split(32)
            out = {}
            for label, p in (("none", None), ("one_user", ["user1@x.org"]), ("user_and_groups", ["user1@x.org", "group2", "group3"])):
                svc._build_filter(**kw, scope_key=("bench", 32), visible_to=p)
                t0 = time.perf_counter()
                for _ in range(200):
                    svc._build_filter(**kw, scope_key=("bench", 32), visible_to=p)
                out[f"fold_us_{label}"] = 1e6 * (time.perf_counter() - t0) / 200
            out["n_scopes"] = len(coll.scope_list)
            return out
        raise ValueError(name)

    print(json.dumps({"ready": True, "lib": os.environ.get("VB200_LIB", "in-tree")}), flush=True)
    for cmd in sys.stdin:
        c = json.loads(cmd)
        if c.get("quit"):
            break
        try:
            res = run_line(c["line"], c["min_s"])
        except Exception as e:
            res = {"error": f"{type(e).__name__}: {e}"}
        res["line"] = c["line"]
        print(json.dumps(res), flush=True)
    VS._drop_collection("acl_bench")


# ---------------------------------------------------------------------------------------------- parent: alternation
LINES = ["none", "k1", "shared4", "shared32", "distinct32", "acl_write", "fold"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--variant", action="append", default=[], metavar="NAME=LIB",
                    help="another library build to compare against (VB200_LIB of a child process); repeatable")
    ap.add_argument("--lines", default=",".join(LINES))
    ap.add_argument("--repeats", type=int, default=3, help="alternations of the builds on line none")
    ap.add_argument("--min-seconds", type=float, default=1.5)
    ap.add_argument("--out", required=True)
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.child:
        return child()
    builds = [("new", None)] + [tuple(v.split("=", 1)) for v in args.variant]
    procs = {}
    for name, lib in builds:
        env = dict(os.environ)
        if lib:
            lib, _, tree = lib.partition(",")
            env["VB200_LIB"] = str(Path(lib).resolve())
            if tree:
                env["ACL_BENCH_TREE"] = str(Path(tree).resolve())
        procs[name] = subprocess.Popen([sys.executable, __file__, "--child", "--out", "-"], env=env, cwd=str(ROOT),
                                       stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True)
        if not procs[name].stdout.readline():
            raise SystemExit(f"build {name}: child process failed to start")

    def ask(name, line):
        p = procs[name]
        p.stdin.write(json.dumps({"line": line, "min_s": args.min_seconds}) + "\n")
        p.stdin.flush()
        r = json.loads(p.stdout.readline())
        r["build"] = name
        print(json.dumps({k: v for k, v in r.items() if k != "digests"}), flush=True)
        return r

    report = {"card_before": card(), "lines": [], "alternation_none": []}
    lines = args.lines.split(",")
    try:
        # line none first on every build (the ACL lines rewrite the scope column of the new build's shard)
        for name, _ in builds:
            report["lines"].append(ask(name, "none"))
        for _ in range(args.repeats):
            for name, _ in builds:
                report["alternation_none"].append(ask(name, "none"))
        for line in lines:
            if line != "none":
                report["lines"].append(ask("new", line))
    finally:
        for p in procs.values():
            try:
                p.stdin.write(json.dumps({"quit": True}) + "\n")
                p.stdin.flush()
            except Exception:
                pass
            p.wait(timeout=300)
    report["card_after"] = card()
    by = {(r["build"], r["line"]): r for r in report["lines"]}
    checks = {}
    for (b, line), r in by.items():
        if b != "new" and line == "none" and ("new", "none") in by:
            checks[f"none_identical_to_{b}"] = r.get("digests") == by[("new", "none")].get("digests")
    if ("new", "k1") in by:
        checks["k1_identical_to_none"] = by[("new", "k1")].get("digests") == by[("new", "none")].get("digests")
    alt = {}
    for r in report["alternation_none"]:
        alt.setdefault(r["build"], []).append(r.get("step_ms"))
    report["alternation_none_step_ms"] = alt
    report["checks"] = checks
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(report, indent=1))
    print(json.dumps({"checks": checks, "alternation_none_step_ms": alt, "card": report["card_before"]}))


if __name__ == "__main__":
    main()
