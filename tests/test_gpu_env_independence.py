"""An index's behaviour depends on its options only, never on the process environment: a process started with
variables that used to retune the library (VB200_DENSE_PATH, VB200_K1F, ...) searches exactly like one started
without them, and the options that lost their A/B runs are unknown keys."""
import json
import os
import subprocess
import sys
from pathlib import Path

import pytest

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parents[1]

# Former tuning variables, each set away from its default.  Only variables that leave results exact: the removed
# perf-triage modes skipped scoring on purpose and are never set here.
FORMER_VARS = {"VB200_DENSE_PATH": "1", "VB200_SPARSE_MS": "0", "VB200_K1F": "0", "VB200_SEG_RATIO": "2",
               "VB200_K2T_STAGES": "2", "VB200_K2_KBOX": "1"}

REMOVED_KEYS = ["dense_wait_sparse", "sel_ctas", "ms_ctas", "ms_stage_ratio", "ms_long_terms", "ms_budget_long",
                "k2t_stages"]

# B = 1 takes the single-pass scan, 8 the resident tensor-core kernel, 320 the query-tiled one.
CHILD = r"""
import json, sys
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
import numpy as np
import _coded, _data
from voitta_rag_b200 import engine

corpus = _data.make_corpus(seed=5, n=20000, dim=128, vocab=2000)
coded = _coded.code_corpus(corpus)
queries = _data.make_queries(seed=6, corpus=corpus, nq=320)
ix = engine.Index(128, device=0)
ix.upsert(coded["dense"], coded["csr"], coded["scope"], coded["created"], coded["modified"])
folders = [f for f, _ in coded["scope_list"]]
flt = engine.Filter(_coded.scope_bits(coded["scope_list"], include=folders[:6]), 2, 1450000000, _coded.TS_MAX)
out = {}
for B in (1, 8, 320):
    Q = np.stack([q for q, _ in queries[:B]])
    SP = [s for _, s in queries[:B]]
    for filtered in (False, True):
        res = ix.search_batch(Q, SP, [flt] if filtered else None, np.zeros(B, np.int32) if filtered else None, limit=10)
        st = ix.stats()
        out[f"B{B}_{'filtered' if filtered else 'unfiltered'}"] = {
            "rows": res.rows.tolist(), "scores": res.scores.tolist(), "counts": res.counts.tolist(),
            "last_dense_path": int(st["last_dense_path"]), "last_launches": int(st["last_launches"])}
ix.close()
with open(sys.argv[2], "w") as f:
    json.dump(out, f)
"""


def run_child(tmp_path, name, extra):
    env = {k: v for k, v in os.environ.items() if not k.startswith("VB200_") or k == "VB200_LIB"}
    env.update(extra)
    env["PYTHONDONTWRITEBYTECODE"] = "1"
    out = tmp_path / f"{name}.json"
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, "-c", CHILD, str(ROOT), str(out)], env=env, cwd=str(ROOT),
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, f"{name} child failed:\n{r.stdout}\n{r.stderr}"
    return json.loads(out.read_text())


def test_former_tuning_variables_change_nothing(tmp_path):
    clean = run_child(tmp_path, "clean", {})
    tuned = run_child(tmp_path, "former_vars", FORMER_VARS)
    assert sorted(clean) == sorted(tuned)
    for case in clean:
        a, b = clean[case], tuned[case]
        assert sum(a["counts"]) > 0, case
        for field in ("last_dense_path", "last_launches", "counts", "rows", "scores"):
            assert a[field] == b[field], f"{case}: {field} depends on the environment"


@pytest.mark.parametrize("key", REMOVED_KEYS)
def test_removed_option_keys_are_unknown(key):
    from voitta_rag_b200 import engine
    ix = engine.Index(16)
    try:
        with pytest.raises(engine.B200Error, match="unknown key"):
            ix.set_option(key, 1)
    finally:
        ix.close()
