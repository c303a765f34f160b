"""What the row selection's reuse across batches (vb_set_option "sel_reuse") saves, and what its miss path costs, on
the cfg4 shard (12.5M x 768, batch 1024, top-100, hybrid RRF, one scope + time filter passing ~50 %).

Every line times run_local + run_fuse with CUDA events on the index's stream, as bench.py does, batch after batch for
at least --seconds of device time (after three warm-up batches), over the same query batches:
  same         one filter for every batch (bench.py's case: the copy is kept from the second batch on)
  alternating  two distinct filters of the same selectivity alternating every batch (every batch copies)
  new          a new filter every batch (every batch copies)
The filters differ only by a shift of their time range (one second per step), so each passes the same ~50 %.

--modes lists the sel_reuse values to run (one index, in order); "default" sets no option, for a build that does not
have it (the parent build, selected with VB200_LIB).  One JSON line per (mode, line), then the card's name, power limit
and max SM clock.  Writes nothing.
    python tools/sel_reuse_bench.py --modes 1,0
    VB200_LIB=<parent build>/libvoitta_b200.so python tools/sel_reuse_bench.py --modes default
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402

import bench  # noqa: E402


def hardware():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = f"nvidia-smi unavailable: {e}"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg4", choices=sorted(bench.WORKLOADS))
    ap.add_argument("--modes", default="1,0", help="comma-separated sel_reuse values, or 'default' (no option set)")
    ap.add_argument("--seconds", type=float, default=1.5, help="device time per line")
    ap.add_argument("--lines", default="same,alternating,new")
    args = ap.parse_args()

    import torch
    from voitta_rag_b200 import engine, synth
    from voitta_rag_b200.sharded import ShardedIndex

    if not torch.cuda.is_available():
        raise SystemExit("sel_reuse_bench.py: no CUDA device")
    cfg = dict(bench.WORKLOADS[args.workload])
    if cfg["sel"] is None:
        raise SystemExit(f"sel_reuse_bench.py: {args.workload} has no filter")
    device = torch.device("cuda", 0)
    torch.cuda.set_device(device)
    ix, keep, _, _ = bench.build_shard(cfg, 0, 1, device, torch, synth, engine)
    sh = ShardedIndex(ix, 0, 1, device=device)
    batches, flt = bench.make_batches(cfg, keep, 1, synth, engine, torch)
    B, limit = cfg["batch"], cfg["limit"]
    hybrid = cfg["fusion"] != "dense"
    kprime = 3 * limit if hybrid else limit
    if hybrid:
        sh.finalize_from_queries([sp for _, sp in batches])
    weighted = [sh.idf_weights(sp) if hybrid else None for _, sp in batches]
    fo = np.zeros(B, np.int32)
    bits, field, lo, hi = flt
    filters = {"same": lambda i: flt, "alternating": lambda i: (bits, field, lo + i % 2, hi + i % 2),
               "new": lambda i: (bits, field, lo + i, hi + i)}

    def one(i, f):
        q, _ = batches[i % len(batches)]
        staged = ix.stage(q, weighted[i % len(batches)], [engine.Filter(*f)], fo, limit=limit, kprime=kprime,
                          fusion=cfg["fusion"], sparse_weight=0.1, apply_idf=False)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(sh.stream):
            ev0.record(sh.stream)
            ix.run_local(None)
            ix.run_fuse(0, None)
            ev1.record(sh.stream)
        if ix.fetch(staged, allow_overflow=True) is None:
            raise SystemExit("sel_reuse_bench.py: candidate overflow")
        st = ix.stats()
        return ev0.elapsed_time(ev1), st["last_launches"], st["last_sel_used"], st["last_sel_rows"]

    for mode in args.modes.split(","):
        if mode != "default":
            ix.set_option("sel_reuse", int(mode))
        for line in args.lines.split(","):
            make = filters[line]
            for i in range(3):
                one(i, make(i))
            ms, launches, n = [], 0, 0
            sel = set()
            while sum(ms) < 1e3 * args.seconds:
                t, l_, used, rows = one(3 + n, make(3 + n))
                ms.append(t)
                launches += l_
                sel.add((used, rows))
                n += 1
            ms = np.asarray(ms)
            print(json.dumps({"workload": args.workload, "sel_reuse": mode, "line": line, "batches": n,
                              "ms_per_batch": round(float(ms.mean()), 4), "ms_median": round(float(np.median(ms)), 4),
                              "ms_min": round(float(ms.min()), 4), "ms_max": round(float(ms.max()), 4),
                              "launches_per_batch": launches / n, "sel_used": sorted({u for u, _ in sel}),
                              "sel_rows_range": [min(r for _, r in sel), max(r for _, r in sel)]}), flush=True)
    print(json.dumps({"hardware": hardware()}), flush=True)
    ix.close()


if __name__ == "__main__":
    main()
