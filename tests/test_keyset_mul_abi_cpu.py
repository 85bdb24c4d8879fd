"""CPU-side check of the keyed scalar multiplication boundary: the plain-C caller of tests/c/keyset_mul_check.c compiles against
include/kyber_b200.h (it is linked and run by the -m gpu suite, tests/test_gpu_keyset_mul.py)."""
import os
import subprocess

from helpers import ROOT


def test_keyset_mul_c_harness_compiles(tmp_path):
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", os.path.join(ROOT, "tests", "c", "keyset_mul_check.c"),
                           "-o", str(tmp_path / "keyset_mul_check.o")])
