"""The PostgreSQL glue (kmer-extension_b200/pgglue/kmer_gpu.c) EXECUTED: its fmgr-V1 SRFs are driven by
tests/c/glue_driver.c through the pgshim with `dna` / `kmer` varlenas of both header forms, next to the reference's own
functions (oracle/_ref) in one process -- or, where oracle/_ref is not built, the C oracle; datums, counts, booleans and
errors must be identical (SURVEY section 8 f1/f2)."""
import subprocess
import sys
from pathlib import Path

import pytest

import golden_util as G

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "kmer-extension_b200"


def build_driver():
    subprocess.run(["make", "-s", "-C", str(PKG / "pgglue")], check=True)
    exe = ROOT / "tests" / "c" / "glue_driver"
    cmd = ["gcc", "-O2", "-std=gnu17", "-Wall", "-I", str(ROOT / "oracle" / "pgshim"), "-I", str(ROOT / "include"),
           str(ROOT / "tests" / "c" / "glue_driver.c"), str(PKG / "pgglue" / "kmer_gpu.o"), "-o", str(exe),
           f"-L{PKG}", "-lkmer_cuda", f"-Wl,-rpath,{PKG}"] + G.expected_side_link_args()
    subprocess.run(cmd, check=True)
    return exe


def test_glue_driver_builds():
    """no GPU needed: glue + driver compile against the pgshim and link against libkmer_cuda.so and the expected side"""
    assert build_driver().exists()


@pytest.mark.gpu
def test_glue_executes_like_the_reference():
    exe = build_driver()
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    sys.stdout.write(r.stdout)
    sys.stderr.write(r.stderr[-2000:])
    assert r.returncode == 0 and "MISMATCH" not in r.stdout, r.stdout[-3000:]
