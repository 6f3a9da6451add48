"""CPU-side checks of the fixed-bases boundary: the C host program compiles against the header
with -Wall -Werror, and without a GPU it fails loudly instead of pretending."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_fixed_bases_c_program_compiles_and_fails_loudly_without_gpu(tmp_path):
    libdir = os.path.join(ROOT, "decaf377_b200")
    if not os.path.exists(os.path.join(libdir, "libdecaf377_b200.so")):
        pytest.skip("library not built")
    exe = tmp_path / "abi_fixed_bases_smoke"
    r = subprocess.run(["gcc", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "abi_fixed_bases_smoke.c"), "-o", str(exe),
                        "-L", libdir, "-ldecaf377_b200", "-Wl,-rpath," + libdir],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: tests/test_gpu_fixed_bases.py runs the program")
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and "check(s) failed" in r.stdout, r.stdout + r.stderr
