"""The C-ABI library loads on a CPU-only box, exports every symbol include/voitta_b200.h declares,
and refuses to compute without a device (no CPU fallback)."""
import ctypes
import re
from pathlib import Path

import pytest

from voitta_rag_b200 import engine

ROOT = Path(__file__).resolve().parents[1]


def declared_symbols():
    text = (ROOT / "include" / "voitta_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(vb_[a-z_0-9]+)\s*\(", text)))


def test_library_exports_exactly_the_declared_symbols():
    lib = engine.load_library()
    syms = declared_symbols()
    assert len(syms) >= 14
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/voitta_b200.h but not exported"
    assert sorted(engine.EXPORTS) == syms
    assert lib.vb_abi_version() == 4


def test_struct_layouts_match_header():
    # sizes implied by the header on LP64
    assert ctypes.sizeof(engine._Filter) == 32
    assert ctypes.sizeof(engine._QueryBatch) == 88
    assert ctypes.sizeof(engine._Result) == 72
    assert ctypes.sizeof(engine._Stats) == 216


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("device present")
    with pytest.raises(engine.B200Error, match="no CPU fallback"):
        engine.Index(64)


def test_product_does_not_import_oracle():
    for p in (ROOT / "voitta-rag_b200").rglob("*.py"):
        src = p.read_text()
        assert "oracle" not in src.replace("no CPU fallback", ""), f"{p} mentions the oracle"
