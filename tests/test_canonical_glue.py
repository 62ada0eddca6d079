"""kmer_gpu_canonical_counts and kmer_gpu_canonical_count_spectrum (kmer-extension_b200/pgglue/kmer_gpu.c) EXECUTED:
tests/c/canonical_driver.c drives both SRFs through the pgshim and compares their rows with the canonical fold of the k-mers
the reference's generate_kmers produces (or the C oracle's, where oracle/_ref is not built), including reverse-complemented
rows, counts beyond the library's histogram and the reference's errors."""
import subprocess
import sys
from pathlib import Path

import pytest

import golden_util as G

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "kmer-extension_b200"


def build_driver():
    subprocess.run(["make", "-s", "-C", str(PKG / "pgglue")], check=True)
    exe = ROOT / "tests" / "c" / "canonical_driver"
    cmd = ["gcc", "-O2", "-std=gnu17", "-Wall", "-I", str(ROOT / "oracle" / "pgshim"), "-I", str(ROOT / "include"),
           str(ROOT / "tests" / "c" / "canonical_driver.c"), str(PKG / "pgglue" / "kmer_gpu.o"), "-o", str(exe),
           f"-L{PKG}", "-lkmer_cuda", f"-Wl,-rpath,{PKG}"] + G.expected_side_link_args()
    subprocess.run(cmd, check=True)
    return exe


def test_canonical_driver_builds():
    """no GPU needed: both SRFs and their driver compile against the pgshim and link against libkmer_cuda.so"""
    assert build_driver().exists()


@pytest.mark.gpu
def test_canonical_srfs_equal_the_folded_group_by():
    exe = build_driver()
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    sys.stdout.write(r.stdout)
    sys.stderr.write(r.stderr[-2000:])
    assert r.returncode == 0 and "MISMATCH" not in r.stdout, r.stdout[-3000:]
    assert r.stdout.count(": ok") == 18
