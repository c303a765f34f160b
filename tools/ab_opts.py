#!/usr/bin/env python
"""A/B runs of index options on ONE resident shard (building a 12.5M-row shard costs more GPU time than timing it).

    python tools/ab_opts.py --workload cfg4 --set "" --set "seg_ratio=8,ms_chunk=1024" --set "dense_compact=0"

Per option set: the options are applied on top of the DEFAULTS given by --base (every key named in any set is reset
to its --base value first), 3 warm-up batches, then --batches batches timed with CUDA events on the launching
stream (the `value` region of bench.py); prints mean / min ms per batch, the dense / sparse chain busy times of a
two-stream timeline batch, and whether the first batch's fused rows equal the first set's."""
from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402


def parse_set(s):
    out = {}
    for kv in filter(None, (x.strip() for x in s.split(","))):
        k, v = kv.split("=", 1)
        out[k] = int(v)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg4", choices=sorted(bench.WORKLOADS))
    ap.add_argument("--set", action="append", default=[], help="comma-separated key=value list; repeatable")
    ap.add_argument("--base", default="", help="values the keys fall back to between sets, e.g. seg_ratio=0,ms_chunk=0")
    ap.add_argument("--batches", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from voitta_rag_b200 import engine, synth

    cfg = dict(bench.WORKLOADS[args.workload])
    device = torch.device("cuda", 0)
    torch.cuda.set_device(device)
    ix, keep, (lo, hi), _ = bench.build_shard(cfg, 0, 1, device, torch, synth, engine)
    batches, flt = bench.make_batches(cfg, keep, 1, synth, engine, torch)
    B, limit = cfg["batch"], cfg["limit"]
    hybrid = cfg["fusion"] != "dense"
    kprime = limit * 3 if hybrid else limit
    filters = None if flt is None else [engine.Filter(*flt)]
    filter_of = None if flt is None else np.zeros(B, np.int32)
    from voitta_rag_b200.sharded import ShardedIndex
    sh = ShardedIndex(ix, 0, 1, device=device)
    if hybrid:
        sh.finalize_from_queries([sp for _, sp in batches])
    weighted = [sh.idf_weights(sp) if hybrid else None for _, sp in batches]
    flush = None
    d_pad = (cfg["dim"] + 63) // 64 * 64
    if (hi - lo) * d_pad * 2 <= 2 * bench.L2_BYTES:
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)

    def stage(i):
        q, _ = batches[i % len(batches)]
        return ix.stage(q, weighted[i % len(batches)], filters, filter_of, limit=limit, kprime=kprime,
                        fusion=cfg["fusion"], sparse_weight=0.1, apply_idf=False)

    def run(i):
        st = stage(i)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(sh.stream):
            if flush is not None:
                flush.fill_(1)
            ev0.record(sh.stream)
            ix.run_local(None)
            ix.run_fuse(0, None)
            ev1.record(sh.stream)
        res = ix.fetch(st, allow_overflow=True)
        if res is None:
            raise OverflowError("candidate list overflow")
        return ev0.elapsed_time(ev1), res

    base = parse_set(args.base)
    sets = [parse_set(s) for s in (args.set or [""])]
    keys = sorted({k for s in sets for k in s} | set(base))
    first_rows = None
    lines = []
    for s in sets:
      try:
        for k in keys:
            ix.set_option(k, s.get(k, base.get(k, 0)))
        ix.set_option("profile", 0)
        ix.set_option("overlap", s.get("overlap", base.get("overlap", 1)))
        for i in range(3):
            run(i)
        ms = []
        res0 = None
        for i in range(args.batches):
            m, res = run(3 + i)
            ms.append(m)
            if i == 0:
                res0 = res
        # batch index 3 of every set is the same batch: compare the fused rows
        rows = np.asarray(res0.rows if hasattr(res0, "rows") else res0[0])
        same = None
        if first_rows is None:
            first_rows = rows.copy()
        else:
            same = bool(np.array_equal(first_rows, rows))
        ix.set_option("profile", 1)
        run(0)
        tl = ix.timeline()
        ix.set_option("profile", 0)

        def busy(names):
            iv = sorted((a_, b_) for n_, _, a_, b_ in tl if n_ in names)
            tot, end = 0.0, -1.0
            for a_, b_ in iv:
                tot += max(0.0, b_ - max(a_, end))
                end = max(end, b_)
            return tot
        # the same batch with the chains serialised: per-launch region times (dense = one region per row segment)
        ix.set_option("profile", 1)
        ix.set_option("overlap", 0)
        run(0)
        tl0 = ix.timeline()
        ix.set_option("profile", 0)
        ix.set_option("overlap", s.get("overlap", base.get("overlap", 1)))
        serial = {n_: [round(b_ - a_, 3) for m_, _, a_, b_ in tl0 if m_ == n_] for n_ in ("dense", "sparse")}
        names = sorted({n_ for n_, _, _, _ in tl})
        span = (max(b_ for _, _, _, b_ in tl) - min(a_ for _, _, a_, _ in tl)) if tl else 0.0
        line = {"set": s, "ms_mean": float(np.mean(ms)), "ms_min": float(np.min(ms)), "qps": B / (float(np.mean(ms)) / 1e3),
                "same_rows_as_first": same, "timeline_span_ms": span,
                "busy_ms": {n_: round(busy((n_,)), 3) for n_ in names}, "launches": int(ix.stats()["last_launches"]), "serial_regions_ms": serial}
        print(json.dumps(line), flush=True)
        lines.append(line)
      except OverflowError as e:
        print(json.dumps({"set": s, "error": str(e)}), flush=True)
    if args.out:
        Path(args.out).write_text("\n".join(json.dumps(l) for l in lines) + "\n")


if __name__ == "__main__":
    main()
