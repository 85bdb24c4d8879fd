"""CPU-side check of the verifier-range share checks: the header declares both entry points, the library exports them, and the
plain-C caller of tests/c/dkg_columns_check.c compiles against include/kyber_b200.h (it is linked and run by the -m gpu suite,
tests/test_gpu_dkg_columns.py)."""
import ctypes
import importlib
import os
import subprocess

from helpers import ROOT

NAMES = ("kb_dkg_verify_columns", "kb_dev_dkg_verify_columns")


def test_dkg_columns_symbols_exported():
    kb = importlib.import_module("kyber-rs_b200")
    L = ctypes.CDLL(kb.LIB_PATH)
    hdr = open(os.path.join(ROOT, "include", "kyber_b200.h")).read()
    for name in NAMES:
        assert name in kb.binding.EXPORTS
        assert hasattr(L, name), name
        assert f"int {name}(" in hdr, name


def test_dkg_columns_c_harness_compiles(tmp_path):
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", os.path.join(ROOT, "tests", "c", "dkg_columns_check.c"),
                           "-o", str(tmp_path / "dkg_columns_check.o")])
