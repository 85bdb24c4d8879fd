"""CPU-side check of the keyed-round boundary: the plain-C caller of tests/c/keyed_round_check.c compiles against
include/kyber_b200.h (it is linked and run by the -m gpu suite, tests/test_gpu_keyed_round.py)."""
import os
import subprocess

from helpers import ROOT


def test_keyed_round_c_harness_compiles(tmp_path):
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", os.path.join(ROOT, "tests", "c", "keyed_round_check.c"),
                           "-o", str(tmp_path / "keyed_round_check.o")])
