"""Throughput of the cfg4 shard (12.5M x 768, hybrid RRF, top-100, batch 1024; bench.py's build_shard / make_batches)
under different filter distributions per batch:

  a      one filter shared by the batch (bench.py's filter, ~50 % selectivity)
  b      1024 separate filters with the content of a (merged into one by the library)
  c      40 distinct filters
  d64, d256, d1024
         that many distinct per-query filters, each a random scope set (synth.scope_filter) with its own date range,
         total selectivity 35-65 %

Every line is warmed, then timed for at least --min-seconds (search_packed: staging + H2D + kernels + D2H + decode,
one batch at a time, 4 query batches in rotation) with the profile option on; one more pass with the two chains
serialised gives per-phase times.  Results are checked: b against a (bit-identical), every line against the other
library builds given with --variant (bit-identical), d1024 against its four 256-query quarters run as separate batches.

Each library build runs in its own child process (VB200_LIB) that keeps its shard resident; the parent process sends
the lines and alternates the builds on line c --repeats times to show the spread.  The card's name, power limit and
SM clock are read before and after.

    python tools/per_query_filters_bench.py --variant parent=/path/to/parent/libvoitta_b200.so --out /tmp/per_query_filters.json
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
sys.path.insert(0, str(ROOT))

LINES = ["a", "b", "c", "d64", "d256", "d1024"]


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else f"nvidia-smi failed: {r.stderr.strip()}"


# ---------------------------------------------------------------------------------------------- child: one library
def child():
    import torch
    import bench
    from voitta_rag_b200 import engine, synth
    cfg = bench.WORKLOADS["cfg4"]
    device = torch.device("cuda", 0)
    ix, keep, (lo, hi), _ = bench.build_shard(cfg, 0, 1, device, torch, synth, engine)
    batches, flt_a = bench.make_batches(cfg, keep, 1, synth, engine, torch)
    batches = batches[:4]
    B, limit, n = cfg["batch"], cfg["limit"], hi - lo
    mask_words = (n + 31) // 32

    def spread(count, seed0):
        out = []
        rng = np.random.RandomState(seed0)
        span = synth.T1 - synth.T0
        for k in range(count):
            t = rng.uniform(0.35, 0.65)
            s = float(np.sqrt(t))
            bits = synth.scope_filter(keep["scope"], s, seed0 * 10_000 + k)
            lo_t = synth.T0 + int(rng.uniform(0.0, 1.0 - s) * span)
            out.append((bits, engine.TS_MODIFIED, lo_t, lo_t + int(s * span)))
        return out

    def line_filters(name):
        if name == "a":
            return [flt_a], np.zeros(B, np.int32)
        if name == "b":
            return [(flt_a[0].copy(),) + tuple(flt_a[1:]) for _ in range(B)], np.arange(B, dtype=np.int32)
        count = 40 if name == "c" else int(name[1:])
        fl = spread(count, seed0=count)
        return fl, (np.random.RandomState(count).permutation(B) % count).astype(np.int32)

    def distinct(fl, fo):
        keys = set()
        for f in np.unique(fo[fo >= 0]):
            bits, field, lo_t, hi_t = fl[f]
            b = np.trim_zeros(np.asarray(bits, np.uint32), "b")
            keys.add((b.tobytes(), field, lo_t, hi_t))
        return len(keys)

    def digest(res):
        h = hashlib.sha1()
        for a in (res.rows, res.scores, res.counts):
            h.update(np.ascontiguousarray(a).tobytes())
        return h.hexdigest()

    cache = {}

    def packs(name):
        if name not in cache:
            fl, fo = line_filters(name)
            gf = [engine.Filter(*f) for f in fl]
            cache[name] = (fl, fo, [ix.pack(q, sp, gf, fo, limit=limit, fusion="rrf") for q, sp in batches])
        return cache[name]

    def run_line(name, min_s):
        fl, fo, ps = packs(name)
        for p in ps:                                           # warm-up of every batch of the line
            ix.search_packed(p)
        digests = [digest(ix.search_packed(p)) for p in ps]
        ix.set_option("profile", 1)
        phase, dev_ms, steps = np.zeros(5), 0.0, 0
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        while True:
            ix.search_packed(ps[steps % len(ps)])
            st = ix.stats()
            phase += [st["last_mask_ms"], st["last_dense_ms"], st["last_sparse_ms"], st["last_select_ms"], st["last_fuse_ms"]]
            dev_ms += st["last_search_ms"]
            steps += 1
            el = time.perf_counter() - t0
            if el >= min_s and steps >= 2 * len(ps):
                break
        ix.set_option("overlap", 0)                            # per-phase times with the chains serialised
        ser = np.zeros(5)
        for p in ps:
            ix.search_packed(p)
            st = ix.stats()
            ser += [st["last_mask_ms"], st["last_dense_ms"], st["last_sparse_ms"], st["last_select_ms"], st["last_fuse_ms"]]
        ix.set_option("overlap", 1)
        ix.set_option("profile", 0)
        st = ix.stats()
        nd = distinct(fl, fo)
        out = {"line": name, "filters_passed": len(fl), "distinct_filters": nd, "steps": steps, "timed_s": el,
               "step_ms": 1e3 * el / steps, "qps": B * steps / el, "device_ms": dev_ms / steps,
               "phase_ms_two_streams": dict(zip(["mask", "dense", "sparse", "select", "fuse"], (phase / steps).round(3).tolist())),
               "phase_ms_serialised": dict(zip(["mask", "dense", "sparse", "select", "fuse"], (ser / len(ps)).round(3).tolist())),
               "mask_bytes": nd * mask_words * 4, "dense_path": int(st["last_dense_path"]), "dense_passes": int(st["last_dense_passes"]),
               "last_sel_used": int(st["last_sel_used"]), "digests": digests}
        if name == "d1024":
            # the same queries as four 256-query batches (at most 256 distinct filters each): identical answers
            same, gf = 0, [engine.Filter(*f) for f in fl]
            q, sp = batches[0]
            full = ix.search_packed(ps[0])
            for k in range(4):
                sl = slice(256 * k, 256 * (k + 1))
                part = ix.search_batch(q[sl], sp[sl], gf, fo[sl], limit=limit, fusion="rrf")
                same += int(sum(np.array_equal(part.rows[i], full.rows[256 * k + i]) and np.array_equal(part.scores[i], full.scores[256 * k + i])
                                for i in range(256)))
            out["quarters_identical_queries"] = same
        return out

    print(json.dumps({"ready": True, "lib": os.environ.get("VB200_LIB", "in-tree")}), flush=True)
    for cmd in sys.stdin:
        c = json.loads(cmd)
        if c.get("quit"):
            break
        try:
            res = run_line(c["line"], c["min_s"])
        except Exception as e:                                 # e.g. a build that cannot run the line
            res = {"line": c["line"], "error": str(e)}
        print(json.dumps(res), flush=True)
    ix.close()


# ---------------------------------------------------------------------------------------------- parent: alternation
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--variant", action="append", default=[], metavar="NAME=LIB",
                    help="another library build to compare against (VB200_LIB of a child process); repeatable")
    ap.add_argument("--lines", default=",".join(LINES))
    ap.add_argument("--repeats", type=int, default=3, help="alternations of the builds on line c")
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
            env["VB200_LIB"] = str(Path(lib).resolve())
        procs[name] = subprocess.Popen([sys.executable, __file__, "--child", "--out", "-"], env=env, cwd=str(ROOT),
                                       stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True)
        ready = procs[name].stdout.readline()
        if not ready:
            raise SystemExit(f"build {name}: child process failed to start")

    def ask(name, line):
        p = procs[name]
        p.stdin.write(json.dumps({"line": line, "min_s": args.min_seconds}) + "\n")
        p.stdin.flush()
        r = json.loads(p.stdout.readline())
        r["build"] = name
        print(json.dumps({k: v for k, v in r.items() if k != "digests"}), flush=True)
        return r

    report = {"card_before": card(), "lines": [], "alternation_c": []}
    try:
        for line in args.lines.split(","):
            for name, _ in builds:
                report["lines"].append(ask(name, line))
        for _ in range(args.repeats):
            for name, _ in builds:
                report["alternation_c"].append(ask(name, "c"))
    finally:
        for p in procs.values():
            try:
                p.stdin.write(json.dumps({"quit": True}) + "\n")
                p.stdin.flush()
            except Exception:
                pass
            p.wait(timeout=120)
    report["card_after"] = card()
    # result checks
    by = {(r["build"], r["line"]): r for r in report["lines"]}
    checks = {}
    if ("new", "a") in by and ("new", "b") in by:
        checks["b_identical_to_a"] = by[("new", "b")].get("digests") == by[("new", "a")].get("digests")
    for (b, line), r in by.items():
        if b != "new" and "digests" in r and ("new", line) in by:
            checks[f"{line}_identical_to_{b}"] = r["digests"] == by[("new", line)].get("digests")
    if ("new", "d1024") in by:
        checks["d1024_quarters_identical_queries"] = by[("new", "d1024")].get("quarters_identical_queries")
    alt = {}
    for r in report["alternation_c"]:
        alt.setdefault(r["build"], []).append(r.get("step_ms"))
    report["alternation_c_step_ms"] = alt
    report["checks"] = checks
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(report, indent=1))
    print(json.dumps({"checks": checks, "alternation_c_step_ms": alt, "card": report["card_before"]}))


if __name__ == "__main__":
    main()
