"""CPU tests of the boundary: libkmer_cuda.so loads, exports every symbol include/kmer_cuda.h
declares, and fails loudly (no CPU fallback) when no CUDA device is present."""
import ctypes as C
import re
from pathlib import Path

import pytest

import conftest  # noqa: F401
from kmer_extension_b200 import api

ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def lib():
    if not api.LIB_PATH.exists():
        import __graft_entry__ as g
        g.build()
    return api.load_library()


def test_header_symbols_exported(lib):
    header = (ROOT / "include" / "kmer_cuda.h").read_text()
    declared = sorted(set(re.findall(r"\b(kmer_cuda_[a-z_0-9]+)\s*\(", header)))
    assert declared, "no declarations parsed"
    for sym in declared:
        assert hasattr(lib, sym), f"{sym} declared in include/kmer_cuda.h but not exported"
    assert sorted(api.ABI_SYMBOLS) == declared


def test_abi_version_and_helpers(lib):
    assert lib.kmer_cuda_abi_version() == 2
    assert lib.kmer_cuda_max_kmers(1000, 1, 21) == 980
    assert lib.kmer_cuda_max_kmers(10, 5, 21) == 0
    assert lib.kmer_cuda_max_kmers(10, 1, 0) == 0
    assert lib.kmer_cuda_max_kmers(10, 1, 33) == 0


def test_struct_layouts_match_header():
    assert C.sizeof(api.KmerCudaError) == 4 + 6 + 160 + 160 + 6 + 8  # int, char[6], 2*char[160], pad to 8, int64
    assert C.sizeof(api.KmerDevResult) == 40
    assert C.sizeof(api.KmerShardPlan) == 72


def test_no_cpu_fallback_without_gpu(lib):
    """Without a device the product path must fail loudly, never compute on the CPU."""
    if lib.kmer_cuda_device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(api.KmerSqlError) as ei:
        api.KmerCuda(0)
    assert ei.value.status == api.KMER_ERR_NO_DEVICE
    assert "no CPU path" in ei.value.message


def test_product_never_imports_oracle():
    """Only tests/, smoke() and bench.py's baseline legs may touch oracle/."""
    for p in (ROOT / "kmer-extension_b200").rglob("*"):
        if p.suffix in {".py", ".cu", ".cuh", ".c", ".h"}:
            txt = p.read_text()
            assert "oracle" not in txt.lower().replace("oracle/pgshim", ""), f"{p} mentions the oracle"


def test_shard_plan_invariants(lib):
    """kmer_cuda_shard_plan is host-only arithmetic: check what the kernels and the exchange rely on."""
    for total in (1, 10_000, 3_000_000, 980_000_000, 7_840_000_000, 80_000_000_000):
        for k in (14, 17, 19, 21, 26, 27, 29, 32):
            for n_ranks in (1, 2, 3, 8, 16):
                for chunks in (1, 2):
                    p = api.KmerShardPlan()
                    assert lib.kmer_cuda_shard_plan_chunked(total, k, n_ranks, chunks, C.byref(p)) == 0
                    assert p.n_ranks == n_ranks and p.chunks_per_rank == chunks and p.k == k
                    assert p.n_buckets == p.buckets_per_rank * n_ranks and p.buckets_per_rank >= 1
                    assert p.cap % 2 == 0 and p.cap >= 64                      # segments start 16-byte aligned
                    assert p.fine_cap % 4 == 0                                  # fine regions are whole 32-byte sectors
                    assert p.rec_bytes == (8 if k <= 26 else 16) and p.recw == (1 if k <= 26 else 2)
                    assert p.recs_bytes_per_peer == p.buckets_per_rank * p.cap * p.rec_bytes
                    assert p.fill_bytes_per_peer == p.buckets_per_rank * 8
                    assert 0 <= p.fine_shift <= 8 and (p.n_buckets << p.fine_shift) < 2 ** 31
                    # every fine bucket holds about 1200 k-mers of the whole job (never more than 2x unless the job is tiny)
                    fine_total = p.n_buckets << p.fine_shift
                    assert fine_total * 1200 >= total
                    # minimizer window: suits the record width, m-mer at most 16 bases, windows fit a record
                    assert p.w in ((4, 6, 8, 9) if k <= 26 else (8, 12, 16))
                    assert p.w != 9 or k <= 22                                  # 9 windows + the k-1 overlap in a 30-base record
                    # the m-mers are fine-grained enough for the buckets (30 per bucket) unless the narrowest window is all that is left
                    fine = 4 ** p.m >= 30 * ((total + 1199) // 1200)
                    assert fine or p.w == (4 if k <= 26 else 8)
                    assert p.even_spread == (0 if fine else 1)                  # too coarse for load-aware buckets: second hash
                    assert p.m == min(16, k - p.w + 1) and p.m >= 2
                    assert 1 <= p.rmax <= 16 and p.rmax + k - 1 <= (30 if k <= 26 else 61)
    bad = api.KmerShardPlan()
    assert lib.kmer_cuda_shard_plan(1000, 13, 2, C.byref(bad)) != 0          # k <= 13 is the dense path
    assert lib.kmer_cuda_shard_plan(1000, 21, 0, C.byref(bad)) != 0
    assert lib.kmer_cuda_shard_plan_chunked(1000, 21, 16, 4, C.byref(bad)) != 0   # at most 32 segments per bucket


def test_shard_plan_window_follows_job_size(lib):
    """Bigger jobs get narrower minimizer windows (longer m-mers): an m-mer cannot be split between buckets."""
    def w(total, k):
        p = api.KmerShardPlan()
        assert lib.kmer_cuda_shard_plan(total, k, 8, C.byref(p)) == 0
        return p.w, p.m
    assert w(980_000_000, 21) == (9, 13)        # 1 GB: 13-base m-mers are enough (82 per bucket)
    assert w(7_840_000_000, 21) == (8, 14)      # 8 GB: 41 14-base m-mers per bucket
    assert w(40_000_000_000, 21) == (6, 16)     # 40 GB
    assert w(9_700_000_000, 31) == (16, 16)     # C3: already 16-base m-mers
    assert w(980_000_000, 27) == (12, 16)       # W=16 would leave 12-base m-mers
    assert w(980_000_000, 17)[0] == 4


def test_bench_reference_arm_prints_one_json_line():
    """`bench.py --impl reference` (the reference's C functions on the host cores) needs no GPU: one JSON line with the
    keys the driver reads; under torchrun every rank but 0 stays silent."""
    import json, os, subprocess, sys
    cmd = [sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--ref-reads", "200",
           "--ref-large-seconds", "0"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "kmers_counted_per_sec_k21" and d["unit"] == "k-mers/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["cpu_baseline"]["kind"] in ("reference", "port")
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    # the reference arm runs on the CUDA arm's config: same workload name, its own sample stated beside it
    assert d["config"]["workload"].startswith("configs[1]: k=21 count over 1 GB") and "200 reads" in d["config"]["sample_per_step"]
    assert d["cpu_baseline"]["sample_scaling"]["largest_sample_that_fits_host_ram_reads"] > 0
    # sized from a calibration pass when --ref-reads is not given; one larger pass beside it
    auto = [sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--ref-seconds", "2",
            "--ref-large-seconds", "3"]
    out2 = subprocess.run(auto, capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out2.returncode == 0, out2.stderr[-2000:]
    d2 = json.loads([ln for ln in out2.stdout.splitlines() if ln.startswith("{")][0])
    sc = d2["cpu_baseline"]["sample_scaling"]
    assert sc["calibration"]["value"] > 0 and d2["value"] > 0
    if "largest_pass" in sc:
        assert sc["largest_pass"]["reads"] <= sc["largest_sample_that_fits_host_ram_reads"]
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and not [ln for ln in out.stdout.splitlines() if ln.startswith("{")]


def test_bench_dump_outputs_do_not_depend_on_table_order(tmp_path):
    """bench.py --dump-outputs: the same table in any order gives the same files, all float64; the sampled codes (64-bit at
    k=32), their counts and the whole table's checksum come back exactly"""
    import importlib.util
    import numpy as np
    import torch
    from oracle import oracle as O
    spec = importlib.util.spec_from_file_location("bench_module", ROOT / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    rng = np.random.default_rng(3)
    keys = np.unique(rng.integers(-(1 << 63), (1 << 63) - 1, 300_000, dtype=np.int64))
    counts = rng.integers(1, 9, keys.size, dtype=np.int64)
    pairs = torch.from_numpy(np.stack([keys, counts], 1))
    outs = []
    for i, p in enumerate((pairs, pairs[torch.randperm(keys.size, generator=torch.Generator().manual_seed(1))])):
        bench.dump_count_table(torch, tmp_path / str(i), p, int(counts.sum()), sample=1 << 12)
        outs.append({f.name: np.load(f) for f in (tmp_path / str(i)).iterdir()})
    assert outs[0].keys() == {"table_sample_codes.npy", "table_sample_counts.npy", "table_stats.npy"}
    for name, a in outs[0].items():
        assert a.dtype == np.float64 and np.array_equal(a, outs[1][name]), name
    hi_lo = outs[0]["table_sample_codes.npy"].astype(np.uint64)
    codes = ((hi_lo[:, 0] << np.uint64(32)) | hi_lo[:, 1]).view(np.int64)
    assert 3000 < codes.size < 6000 and np.all(codes[1:] > codes[:-1])
    at = np.searchsorted(keys, codes)
    assert np.array_equal(keys[at], codes) and np.array_equal(outs[0]["table_sample_counts.npy"], counts[at])
    n, n_kmers, cnt, hi, lo = (int(x) for x in outs[0]["table_stats.npy"])
    assert n == keys.size and n_kmers == cnt == int(counts.sum())
    assert (hi << 32 | lo) == O.np_table_checksum(keys.view(np.uint64), counts.astype(np.uint64))


@pytest.mark.gpu
def test_bench_dump_outputs_hold_the_counted_table(tmp_path):
    """`bench.py --dump-outputs` on the GPU: the files appear, their statistics are those of the table the JSON line reports,
    and the sample -- the whole table while it has at most 2^20 groups -- is the oracle's GROUP BY of the same seeded reads"""
    import json, subprocess, sys
    import numpy as np
    from kmer_extension_b200 import datagen
    from oracle import oracle as O
    reads = 1000                                   # 980 000 windows: under the 2^20 groups of the sample
    cmd = [sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--reads", str(reads), "--steps", "2", "--warmup", "3",
           "--no-e2e", "--no-cpu", "--no-secondary", "--dump-outputs", str(tmp_path)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    assert d["steps"] == 2 and d["parity"]["checksum_ok"] and d["parity"]["count_ok"]
    flat, off = datagen.synth_reads(2, reads, 1000)
    keys, counts, n = O.np_count(flat, off, 21)
    s, _ = O.COracle().multiset_checksum(flat, off, 21)
    stats = [int(x) for x in np.load(tmp_path / "table_stats.npy")]
    assert stats == [keys.size, n, n, s >> 32, s & 0xffffffff] and d["config"]["n_distinct_rank0"] == keys.size
    hi_lo = np.load(tmp_path / "table_sample_codes.npy").astype(np.uint64)
    assert np.array_equal((hi_lo[:, 0] << np.uint64(32)) | hi_lo[:, 1], keys)
    assert np.array_equal(np.load(tmp_path / "table_sample_counts.npy"), counts.astype(np.float64))


def test_pg_regress_suite_is_generated_from_the_kats():
    """kmer-extension_b200/pgglue/regress/{sql,expected} are what tools/make_pg_regress.py derives from tests/golden/kat.json"""
    import subprocess, sys
    reg = ROOT / "kmer-extension_b200" / "pgglue" / "regress"
    before = ((reg / "sql" / "kmer_kat.sql").read_text(), (reg / "expected" / "kmer_kat.out").read_text())
    subprocess.run([sys.executable, str(ROOT / "tools" / "make_pg_regress.py")], check=True, capture_output=True)
    after = ((reg / "sql" / "kmer_kat.sql").read_text(), (reg / "expected" / "kmer_kat.out").read_text())
    assert before == after
    assert "kmer_gpu_counts" in after[0] and "tacg |     1" in after[1]


def test_every_library_call_of_the_python_host_side_has_argtypes():
    """ctypes passes a bare Python int as a 32-bit C int: a device pointer handed to a function without argtypes is truncated
    (found on the GPU: kmer_cuda_dev_synth_reads wrote through half a pointer).  Every kmer_cuda_* function the Python host side
    calls with arguments must declare them."""
    import re
    from kmer_extension_b200 import api
    lib = api.load_library()
    called = set()
    for f in ("api.py", "sharded.py"):
        called |= set(re.findall(r"lib\.(kmer_cuda_\w+)\(", (ROOT / "kmer-extension_b200" / f).read_text()))
    called |= set(re.findall(r"lib\.(kmer_cuda_\w+)\(", (ROOT / "bench.py").read_text()))
    no_args = {"kmer_cuda_abi_version", "kmer_cuda_device_count"}
    missing = sorted(n for n in called - no_args if getattr(lib, n).argtypes is None)
    assert not missing, f"no argtypes: {missing}"


def test_multi_and_generator_entry_points_reject_bad_arguments_without_touching_a_device(lib):
    """NULL handles / missing out-pointers come back as KMER_ERR_BAD_ARGUMENT, and a device list cannot be opened without a
    GPU (KMER_ERR_NO_DEVICE: the multi-device handle has no CPU path either)."""
    BAD = 16  # KMER_ERR_BAD_ARGUMENT, include/kmer_cuda.h
    hdr = (ROOT / "include" / "kmer_cuda.h").read_text()
    assert re.search(r"KMER_ERR_BAD_ARGUMENT\s*=\s*16", hdr)
    vp, u64 = C.c_void_p, C.c_uint64
    lib.kmer_cuda_multi_submit_match.argtypes = [vp, C.c_int, vp, vp, vp, u64, C.c_int, vp, C.c_uint32, vp, vp, vp]
    lib.kmer_cuda_multi_submit_count.argtypes = [vp, vp, vp, u64, C.c_int, vp, vp, vp]
    lib.kmer_cuda_init_multi.argtypes = [C.POINTER(vp), C.POINTER(C.c_int), C.c_int]
    bits, wpr, hits = vp(), u64(), vp()
    assert lib.kmer_cuda_multi_submit_match(None, 0, None, None, None, 0, 12, None, 0, C.byref(bits), C.byref(wpr), C.byref(hits)) == BAD
    assert lib.kmer_cuda_multi_submit_count(None, None, None, 0, 21, None, None, None) == BAD
    assert lib.kmer_cuda_dev_synth_reads(None, 1, 0, 1, 1, None, None, None) == BAD
    h = vp()
    assert lib.kmer_cuda_init_multi(C.byref(h), None, 0) == BAD
    assert lib.kmer_cuda_init_multi(C.byref(h), (C.c_int * 17)(), 17) == BAD
    if lib.kmer_cuda_device_count() == 0:
        devs = (C.c_int * 2)(0, 1)
        rc = lib.kmer_cuda_init_multi(C.byref(h), devs, 2)
        assert rc == api.KMER_ERR_NO_DEVICE and not h.value
        e = lib.kmer_cuda_last_error(None).contents
        assert b"no CPU path" in e.message


def test_committed_sass_counts_belong_to_the_built_library():
    """bench.py's secondary.match_c4.int32 multiplies the static instruction counts of match_table_kernel's round loop
    (profiles/r02_match_table_sass_counts.json) by the trip count: the committed counts must be those of the library as built
    from the current sources."""
    import importlib.util
    import json
    import shutil
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    spec = importlib.util.spec_from_file_location("sass_loop_count", ROOT / "tools" / "sass_loop_count.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    committed = json.loads((ROOT / "profiles" / "r02_match_table_sass_counts.json").read_text())
    now = mod.loop_counts(committed["function"])
    assert now["instructions"] == committed["instructions"] and now["by_pipe"] == committed["by_pipe"], \
        "match.cu changed: run `python tools/sass_loop_count.py` and commit profiles/r02_match_table_sass_counts.json"
    assert committed["by_pipe"]["alu"] > committed["instructions"] // 2      # the loop is LOP3 / SHF work
    assert committed["pair_tests_per_loop_trip"] == 32 * 1024
