"""Every entry point of the C ABI is exercised by the suite: a symbol bound in _lib.SIGNATURES (every symbol
include/idf_b200.h declares) must be named by some test file, or be listed below with the Python wrapper that calls it
and the test that drives that wrapper.  A new entry point without a test fails here instead of going unnoticed."""
import re
from pathlib import Path

from infodiffusion_b200 import _lib

ROOT = Path(__file__).resolve().parent.parent
TESTS = ROOT / "tests"

# symbol -> (module that calls it, test that drives that module: "file::function")
VIA_WRAPPER = {
    "idf_clip_adamw": ("infodiffusion_b200/optim.py", "test_gpu_ops.py::test_clip_adamw_matches_torch"),
    "idf_mmd_fwd_bwd": ("infodiffusion_b200/utils.py", "test_gpu_ops.py::test_mmd_against_oracle_and_golden"),
}


def _named(symbol: str, text: str) -> bool:
    return re.search(rf"\b{re.escape(symbol)}\b", text) is not None


def test_every_entry_point_is_named_by_a_test():
    me = Path(__file__).resolve()
    text = "\n".join(p.read_text() for p in sorted(TESTS.rglob("*.py")) if p.resolve() != me)
    missing = [s for s in _lib.SIGNATURES if s not in VIA_WRAPPER and not _named(s, text)]
    assert not missing, f"C-ABI entry points no test calls: {missing}"


def test_wrapper_map_points_at_real_callers_and_tests():
    for symbol, (module, test_id) in VIA_WRAPPER.items():
        assert symbol in _lib.SIGNATURES, f"{symbol} is not a C-ABI entry point"
        assert _named(symbol, (ROOT / module).read_text()), f"{module} does not call {symbol}"
        fname, test = test_id.split("::")
        assert re.search(rf"^def {test}\(", (TESTS / fname).read_text(), re.M), f"{test_id} does not exist"
