"""The planner hook of the PostgreSQL glue (kmer-extension_b200/pgglue/kmer_gpu_hook.c, SURVEY 8 f4) run on hand-built analyzed
Query trees through the pgshim's node stand-ins (tests/c/hook_driver.c): the reference's stock counting queries
(kmer-tests.sql:1162-1181) become a function scan on kmer_gpu_counts, everything else reaches the planner untouched; on a GPU
the rewritten tree is executed and must return what the original query returns with the reference's own generate_kmers
(oracle/_ref), or, where that is not built, with the C oracle's."""
import subprocess
import sys
from pathlib import Path

import pytest

import golden_util as G

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "kmer-extension_b200"


def build_driver():
    subprocess.run(["make", "-s", "-C", str(PKG / "pgglue")], check=True)
    exe = ROOT / "tests" / "c" / "hook_driver"
    cmd = ["gcc", "-O2", "-std=gnu17", "-Wall", "-I", str(ROOT / "oracle" / "pgshim"), "-I", str(ROOT / "include"),
           str(ROOT / "tests" / "c" / "hook_driver.c"), str(ROOT / "oracle" / "pgshim_nodes.c"), str(PKG / "pgglue" / "kmer_gpu_hook.o"),
           str(PKG / "pgglue" / "kmer_gpu.o"), "-o", str(exe), f"-L{PKG}", "-lkmer_cuda", f"-Wl,-rpath,{PKG}"] + G.expected_side_link_args()
    subprocess.run(cmd, check=True)
    return exe


def test_hook_rewrites_the_stock_count_queries_and_nothing_else():
    """no GPU needed: matcher + rewrite on the three stock shapes, their ORDER BY / LIMIT variants and 18 queries that must
    stay untouched"""
    exe = build_driver()
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    sys.stdout.write(r.stdout)
    assert r.returncode == 0 and "MISMATCH" not in r.stdout and "all ok" in r.stdout, r.stdout[-3000:] + r.stderr[-1000:]
    assert r.stdout.count(" ok\n") >= 25


@pytest.mark.gpu
def test_rewritten_plan_executes_like_the_original_query():
    exe = build_driver()
    r = subprocess.run([str(exe), "--exec"], capture_output=True, text=True, timeout=600)
    sys.stdout.write(r.stdout)
    sys.stderr.write(r.stderr[-2000:])
    assert r.returncode == 0 and "MISMATCH" not in r.stdout and "rewritten plan on the GPU" in r.stdout, r.stdout[-3000:]
