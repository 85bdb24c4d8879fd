"""CPU-side check of the round-check mode boundary: the header declares it, the library exports it, and the plain-C caller of
tests/c/round_batched_check.c compiles against include/kyber_b200.h (it is linked and run by the -m gpu suite,
tests/test_gpu_round_batched.py)."""
import ctypes
import importlib
import os
import subprocess

from helpers import ROOT


def test_round_check_symbols_exported():
    kb = importlib.import_module("kyber-rs_b200")
    L = ctypes.CDLL(kb.LIB_PATH)
    for name in ("kb_ctx_set_round_check", "kb_ctx_round_fallbacks"):
        assert name in kb.binding.EXPORTS
        assert hasattr(L, name), name
    hdr = open(os.path.join(ROOT, "include", "kyber_b200.h")).read()
    assert "KB_ROUND_CHECK_EXACT = 0" in hdr and "KB_ROUND_CHECK_BATCHED = 1" in hdr
    assert kb.binding.ROUND_CHECK == {"exact": 0, "batched": 1}


def test_round_batched_c_harness_compiles(tmp_path):
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", os.path.join(ROOT, "tests", "c", "round_batched_check.c"),
                           "-o", str(tmp_path / "round_batched_check.o")])
