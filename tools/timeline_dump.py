#!/usr/bin/env python
"""Print the CUDA-event timeline (every timed region, per stream) of one batch of a bench workload on a resident shard:
python tools/timeline_dump.py --workload cfg4 --set seg_ratio=8"""
import argparse, json, sys
from pathlib import Path
ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import numpy as np
import torch
import bench
from voitta_rag_b200 import engine, synth
from voitta_rag_b200.sharded import ShardedIndex

ap = argparse.ArgumentParser()
ap.add_argument("--workload", default="cfg4")
ap.add_argument("--set", action="append", default=[])
args = ap.parse_args()
cfg = dict(bench.WORKLOADS[args.workload])
device = torch.device("cuda", 0)
torch.cuda.set_device(device)
ix, keep, (lo, hi), _ = bench.build_shard(cfg, 0, 1, device, torch, synth, engine)
sh = ShardedIndex(ix, 0, 1, device=device)
batches, flt = bench.make_batches(cfg, keep, 1, synth, engine, torch)
filters = None if flt is None else [engine.Filter(*flt)]
B = cfg["batch"]
filter_of = np.zeros(B, np.int32) if flt is not None else None
hybrid = cfg["fusion"] != "dense"
limit = cfg["limit"]
kprime = limit * 3 if hybrid else limit
if hybrid:
    sh.finalize_from_queries([sp for _, sp in batches])
weighted = [sh.idf_weights(sp) if hybrid else None for _, sp in batches]


def run(i):
    q, _ = batches[i % len(batches)]
    st = ix.stage(q, weighted[i % len(batches)], filters, filter_of, limit=limit, kprime=kprime, fusion=cfg["fusion"], sparse_weight=0.1, apply_idf=False)
    with torch.cuda.stream(sh.stream):
        ix.run_local(None)
        ix.run_fuse(0, None)
    return ix.fetch(st, allow_overflow=True)


for sset in (args.set or [""]):
    for kv in filter(None, sset.split(",")):
        k, v = kv.split("=")
        ix.set_option(k, int(v))
    for i in range(4):
        run(i)
    ix.set_option("profile", 1)
    run(0)
    tl = ix.timeline()
    ix.set_option("profile", 0)
    print("==", sset or "(defaults)")
    for name, big, a, b in sorted(tl, key=lambda r: r[2]):
        print(f"  {a:8.3f} -> {b:8.3f}  ({b - a:7.3f} ms)  {name}{' *' if big else ''}")
