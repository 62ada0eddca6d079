#!/usr/bin/env python
"""bench.py -- k-mers counted per second (whole job) at k=21 on synthetic 1 kb reads.

    python bench.py --gpus 1 --steps K --warmup W            # this repository's CUDA path
    python bench.py ... --dump-outputs DIR                    # + the last timed step's (k-mer, count) table as .npy files
                                                              # (seeded inputs: two builds compare output for output)
    python bench.py --impl reference --steps K --warmup W     # the reference's C functions on the host cores: every step a
                                                              # bounded sample of the same workload, sized from a calibration
                                                              # pass (--ref-seconds), + one larger pass reported beside it

One "step" = one full pass of the hot path (generate_kmers over every row + GROUP BY count) over one
batch.  N=1 workload = BASELINE.json configs[1]: k=21 count over 1 GB of synthetic DNA
(1 000 000 reads x 1 000 bases, i.i.d. uniform ACGT, seed 2 -- kmer-extension_b200/datagen.py restates
the reference's data_generator.py distribution).

value : k-mers/s with the input already resident in HBM (CUDA events around K steps, max over ranks)
e2e   : the same metric through the host-buffer C ABI call kmer_cuda_submit_count (pinned host input,
        H2D + kernels + D2H of the (k-mer,count) table inside the timed region)
roofline     : dominant kernel, algorithmic bytes / its own CUDA-event duration vs MEASURED_PEAKS.json
roofline_step: whole step against SURVEY section 8(d)'s B_alg = N_bases + 16*D
cpu_baseline : the reference's own C code (oracle/_ref, PG executor emulated) on the host cores,
               bounded sample, rank 0 only
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "kmers_counted_per_sec_k21"
UNIT = "k-mers/s"
READ_LEN = 1000
K = 21


def load_pkg():
    import __graft_entry__ as g
    g.load_package()
    from kmer_extension_b200 import api, datagen
    return g, api, datagen


def workload_name(config: str, k: int, n_rows: int) -> str:
    """config.workload of BOTH arms (the reference arm runs bounded samples of the same workload)."""
    gb = n_rows * READ_LEN / 1e9
    return {"c2": f"configs[1]: k={k} count over {gb:.3g} GB synthetic DNA per GPU ({n_rows} reads x {READ_LEN}, seed 2+rank)",
            "c3": f"configs[2]: k=31 count over 10 GB synthetic DNA in total, {n_rows} reads x {READ_LEN} per GPU (seed 3+rank)",
            "c2x10": f"north-star shape: k=21 count over 10 GB synthetic DNA in total, {n_rows} reads x {READ_LEN} per GPU (seed 2+rank)"}[config]


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"



# ------------------------------------------------------------------------------------------------------------------
# parity at config scale (outside every timed region): the GROUP BY table must hold exactly the multiset of windows
# generate_kmers yields.  CPU side: the C oracle's order-independent checksum of the INPUT rows, sum of mix64(code) over
# all windows mod 2^64 (oracle/kmer_oracle.c orc_multiset_checksum, validated against np_count in tests/test_oracle.py).
# GPU side (torch, harness only): sum over groups of count * mix64(code), plus sum of counts and key uniqueness by a sort.
M64 = (1 << 64) - 1


def _s64(v):
    v &= M64
    return v - (1 << 64) if v >> 63 else v


def mix64_torch(torch, x):
    """murmur3 finaliser on int64 tensors (two's complement wrap == uint64 arithmetic)."""
    lo31 = (1 << 31) - 1
    x = x ^ ((x >> 33) & lo31)
    x = x * _s64(0xff51afd7ed558ccd)
    x = x ^ ((x >> 33) & lo31)
    x = x * _s64(0xc4ceb9fe1a85ec53)
    x = x ^ ((x >> 33) & lo31)
    return x


def table_checksum(torch, keys, counts=None, chunk=1 << 26):
    """(sum count*mix64(key) mod 2^64, sum of counts) of a device table; counts=None means every count is 1."""
    tot, cnt = 0, 0
    n = keys.numel()
    for i in range(0, n, chunk):
        k = keys[i:i + chunk]
        m = mix64_torch(torch, k)
        if counts is not None:
            c = counts[i:i + chunk]
            m = m * c
            cnt += int(c.sum().item())
        else:
            cnt += k.numel()
        tot = (tot + int(m.sum().item())) & M64
    return tot, cnt


def keys_unique(torch, keys):
    if keys.numel() < 2:
        return True
    if keys.numel() >= (1 << 30):        # torch.sort takes at most INT_MAX elements: equal keys share their low bits, sort by piece
        pieces = 1
        while keys.numel() // pieces >= (1 << 29):
            pieces *= 2
        low = keys & (pieces - 1)
        return all(keys_unique(torch, keys[low == r]) for r in range(pieces))
    s, _ = torch.sort(keys)
    return not bool((s[1:] == s[:-1]).any().item())


def dump_count_table(torch, out_dir, pairs, n_kmers, suffix="", sample=1 << 20, chunk=1 << 26):
    """--dump-outputs: the (k-mer, count) table one count call returned, as float64 .npy files two builds can be compared by.
    The table comes back in hash order with up to one group per window (16 GB at 1 GB of random reads), so what is written is
    the groups whose mix64(code) falls under a threshold sized for about `sample` groups -- the same groups whatever the
    order -- sorted by code, plus the size and checksum of the whole table.  A code has 2k bits: it is stored as its high and
    low 32-bit halves, which float64 holds exactly; so is the 64-bit checksum."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    keys, counts = pairs[:, 0], pairs[:, 1]
    n = keys.numel()
    thr = min(1 << 24, -(-(sample << 24) // max(n, 1)))          # compared with the top 24 bits of mix64(code)
    picked = [pairs[i:i + chunk][((mix64_torch(torch, keys[i:i + chunk]) >> 40) & 0xffffff) < thr] for i in range(0, n, chunk)]
    picked = torch.cat(picked) if picked else pairs[:0]
    picked = picked[torch.argsort(picked[:, 0])][:2 * sample].cpu().numpy()
    codes = picked[:, 0].astype(np.uint64)
    tot, cnt = table_checksum(torch, keys, counts)
    np.save(out / f"table_sample_codes{suffix}.npy", np.stack([codes >> np.uint64(32), codes & np.uint64(0xffffffff)], 1).astype(np.float64))
    np.save(out / f"table_sample_counts{suffix}.npy", picked[:, 1].astype(np.float64))
    # distinct k-mers, k-mers counted, sum of the counts, checksum (high, low 32 bits) -- see table_checksum
    np.save(out / f"table_stats{suffix}.npy", np.array([n, n_kmers, cnt, tot >> 32, tot & 0xffffffff], dtype=np.float64))


def input_checksum(flat, off, k):
    from oracle import oracle as O
    return O.COracle().multiset_checksum(flat, off, k)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def mark_begin(self):
        self.t_begin = time.time()

    def mark_end(self):
        self.t_end = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        t0, t1 = getattr(self, "t_begin", 0.0), getattr(self, "t_end", float("inf"))
        inside = [ln for (ts, ln) in self.lines if t0 - 0.005 <= ts <= t1 + 0.03]
        window = "timed region"
        if len(inside) < 2:          # a timed region shorter than two sampling periods: take the warm-up steps as well
            inside = [ln for (ts, ln) in self.lines if ts <= t1 + 0.03]
            window = "warm-up + timed region (same load)"
        sm, smax, reasons = [], [], set()
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


def cpu_reference_run(datagen, n_reads: int, threads: int, steps: int, warmup: int):
    """The reference's own kmer.c (oracle/_ref) or, failing that, the C port, on the host cores."""
    from oracle import oracle as O
    flat, off = datagen.synth_reads(2, n_reads, READ_LEN)
    if O.REF_SO.exists():
        R = O.Ref()
        kind = "reference"
        run = lambda: R.count(flat, off, K, threads=threads)[2]
    else:
        O.build(ref=False)
        Cc = O.COracle()
        kind, threads = "port", 1
        run = lambda: Cc.count(flat, off, K)[2]
    for _ in range(warmup):
        run()
    t0 = time.perf_counter()
    n = 0
    for _ in range(steps):
        n += run()
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": UNIT, "cores": threads, "kind": kind,
            "sample": f"{n_reads} reads x {READ_LEN} bases (seed 2 prefix of the workload), k={K}, "
                      f"generate_kmers + hash aggregate (Partial per thread + serial Finalize), {steps} pass(es)",
            "seconds": dt, "steps": steps}


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def available_host_ram() -> int:
    """what this process may still allocate: /proc/meminfo's MemAvailable, or less under a cgroup limit (v2 or v1)"""
    import psutil
    avail = int(psutil.virtual_memory().available)
    for lim, cur in (("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory.current"),
                     ("/sys/fs/cgroup/memory/memory.limit_in_bytes", "/sys/fs/cgroup/memory/memory.usage_in_bytes")):
        try:
            limit = Path(lim).read_text().strip()
            if limit != "max" and int(limit) < (1 << 60):
                avail = min(avail, max(int(limit) - int(Path(cur).read_text().strip()), 0))
        except (OSError, ValueError):
            pass
    return avail


def ref_sample_plan(args, rate_small: float, threads: int):
    """How many reads one step of the reference arm counts: sized from a calibration pass so that warm-up + steps take about
    --ref-seconds, and bounded by what the executor stand-in's hash table can hold in this host's RAM."""
    kmers_per_read = READ_LEN - K + 1
    avail = available_host_ram()
    # measured on the reference driver (oracle/ref_driver.c): ~155 B of RSS per group at k=21 (entry + ASCII key + per-thread
    # partial tables + the merged table), random DNA has one group per window
    bytes_per_group = 160
    fit_reads = int(0.6 * avail / bytes_per_group / kmers_per_read)
    if args.ref_reads > 0:
        return args.ref_reads, fit_reads, avail
    per_step = min(max(args.ref_seconds / max(args.steps + args.warmup, 1), 0.5), 30.0)
    n = int(0.8 * rate_small * per_step / kmers_per_read)     # 0.8: the rate drops as the table outgrows the caches
    return max(2000, min(n, fit_reads, args.reads)), fit_reads, avail


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path, all host threads.  Every step counts a bounded
    sample (a prefix of the same seeded workload); the sample is sized from a calibration pass, and ONE more pass over the
    largest sample that is affordable in time and host RAM is reported beside it so that the per-k-mer rate is not
    extrapolated from a table that fits the caches."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    _, api, datagen = load_pkg()
    threads = host_threads()
    reads_per_gpu = args.reads if args.config == "c2" else 10_000_000 // max(args.gpus, 1)   # as the CUDA arm splits the job
    cal = cpu_reference_run(datagen, 2000, threads, 1, 0)
    n_reads, fit_reads, avail = ref_sample_plan(args, cal["value"], threads)
    r = cpu_reference_run(datagen, n_reads, threads, args.steps, args.warmup)
    kmers_per_read = READ_LEN - K + 1
    scaling_info = {"calibration": {"reads": 2000, "value": cal["value"]},
                    "host_ram_available_bytes": int(avail),
                    "largest_sample_that_fits_host_ram_reads": int(fit_reads),
                    "whole_workload_reads": int(args.reads),
                    "whole_workload_fits_host_ram": bool(fit_reads >= args.reads)}
    if args.ref_large_seconds > 0:
        # half of what fits: the per-group figure is a measurement at k=21 on one box, not a guarantee
        n_large = int(min(fit_reads // 2, args.reads, r["value"] * args.ref_large_seconds / kmers_per_read))
        if n_large > 2 * n_reads:
            big = cpu_reference_run(datagen, n_large, threads, 1, 0)
            scaling_info["largest_pass"] = {"reads": n_large, "value": big["value"], "unit": UNIT, "seconds": big["seconds"],
                                            "what": "one untimed-by-the-driver pass over the largest sample affordable in "
                                                    f"{args.ref_large_seconds:.0f} s and in host RAM; not the line's value"}
    cpu = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
    cpu["sample_scaling"] = scaling_info
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * r["seconds"] / max(args.steps, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": workload_name(args.config, K, reads_per_gpu), "k": K, "read_len": READ_LEN,
                       "reads_per_gpu": reads_per_gpu, "algo": 0,
                       "sample_per_step": f"{n_reads} reads x {READ_LEN} bases (prefix of the workload, seed 2)"},
            "cpu_baseline": cpu,
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_secondary(args):
    """Secondary single-GPU measurements of the other rows of the path (not the headline line):
       extract  : generate_kmers over 1 GB, k=21              B_alg = N + 8*n_kmers
       match_c5 : equals + starts_with in ONE pass over M 32-mers (configs[4])   B_alg = 8*M + 2*M/8
       match_c4 : contains, 1000 IUPAC patterns (k=12) x M k-mers (configs[3])   B_alg = 8*M + 16*P + P*M/8"""
    import torch
    g, api, datagen = load_pkg()
    torch.cuda.set_device(0)
    eng = api.KmerCuda(0)
    peak, peak_src = measured_peaks()
    stream = torch.cuda.current_stream()

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps

    if args.workload == "extract":
        n_rows = args.reads
        flat, off = datagen.synth_reads(2, n_rows, READ_LEN)
        n_bases = int(off[-1])
        d_seq = torch.from_numpy(np.concatenate([flat, np.zeros(64, np.uint8)])).cuda()
        d_off = torch.from_numpy(off.astype(np.int64)).cuda()
        n_k = eng.max_kmers(n_bases, n_rows, K)
        d_codes = torch.empty(n_k, dtype=torch.int64, device="cuda")

        def fn():
            eng.dev_extract(d_seq, n_bases, d_off, n_rows, K, d_codes, stream=stream)
            eng.dev_finish(stream)
        ms = timed(fn)
        alg = n_bases + 8 * n_k
        units, unit, metric = n_k, "k-mers/s", "kmers_extracted_per_sec_k21"
        wl = f"generate_kmers over {n_bases / 1e9:.3g} GB ({n_rows} reads x {READ_LEN}), k={K}"
    else:
        if args.workload == "match_c5":
            m, k, P = args.match_m or 1_000_000_000, 32, 2
            col = datagen.synth_kmer_codes(5, m, k)
            txt = "".join("acgt"[(int(col[0]) >> (2 * (31 - j))) & 3] for j in range(32))
            consts, ops = [txt, txt[:8]], [api.OP_EQUALS, api.OP_STARTS_WITH]
            alg = 8 * m + 2 * ((m + 7) // 8)
            wl = f"configs[4]: equals + starts_with(8-base prefix) in one pass over {m:.3g} 32-mers"
        else:
            m, k, P = args.match_m or 100_000_000, 12, 1000
            col = datagen.synth_kmer_codes(4, m, k)
            consts, ops = datagen.synth_qkmers(4, P, k, with_n=True), None
            alg = 8 * m + 16 * P + P * ((m + 7) // 8)
            wl = f"configs[3]: contains, {P} IUPAC patterns (k=12, 15-letter alphabet incl. N) x {m:.3g} k-mers, full bit matrix"
        d_col = torch.from_numpy(col.view(np.int64)).cuda()
        wpr = (m + 31) // 32
        d_bits = torch.empty(P * wpr, dtype=torch.int32, device="cuda")
        d_hits = torch.empty(P, dtype=torch.int64, device="cuda")
        op = api.OP_CONTAINS if args.workload == "match_c4" else api.OP_EQUALS

        def fn():
            eng.dev_match(op, d_col, m, k, consts, d_bits, d_hits, ops=ops, stream=stream)
            eng.dev_finish(stream)
        ms = timed(fn)
        units, unit, metric = m * P, "pair-tests/s", f"{args.workload}_pair_tests_per_sec"
    ach = alg / (ms * 1e-3) / 1e9
    line = {"metric": metric, "value": units / (ms * 1e-3), "unit": unit, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": wl, "secondary": True},
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                         "alg_bytes_per_launch": alg, "peak_source": peak_src},
            "gpu_launches": int(eng.launches)}
    print(json.dumps(line), flush=True)
    eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--reads", type=int, default=1_000_000, help="reads per GPU (1 kb each); default = 1 GB")
    ap.add_argument("--algo", type=int, default=0, help="0 auto, 1 dense, 2 hash, 3 minimizer partition")
    ap.add_argument("--ref-reads", type=int, default=0, help="reads per step of the reference arm (0 = sized from a calibration pass "
                                                             "so that the run takes about --ref-seconds)")
    ap.add_argument("--ref-seconds", type=float, default=120.0, help="time budget of the reference arm's warm-up + timed steps")
    ap.add_argument("--ref-large-seconds", type=float, default=45.0,
                    help="reference arm: one extra pass over the largest sample affordable in this many seconds (0 = skip)")
    ap.add_argument("--cpu-reads", type=int, default=20000, help="sample size of the cpu_baseline leg")
    ap.add_argument("--workload", default="count", choices=["count", "extract", "match_c4", "match_c5"],
                    help="count = the headline (configs[1]); the others are secondary parity-config measurements")
    ap.add_argument("--match-m", type=int, default=0, help="k-mers in the match workloads (default: the config's size)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the short extract / match measurements")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle checksum of the result tables (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the (k-mer, count) table of the last timed step to DIR as .npy files (a seeded sample of the "
                         "groups plus the whole table's size and checksum, see dump_count_table)")
    ap.add_argument("--devgen", action="store_true", help="generate the reads in HBM (kmer_cuda_dev_synth_reads: one seeded table, every rank "
                                                          "its own row range) instead of on the host with numpy")
    ap.add_argument("--k", type=int, default=21, help="k-mer length of the count workload (default: the headline's 21)")
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c2x10"],
                    help="c2 = BASELINE configs[1] (default; weak scaling, --reads per GPU); c3 = configs[2]: k=31 over 10 GB in total, "
                         "strong-scaled over the GPUs; c2x10 = the north star's shape: k=21 over 10 GB in total")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "count"):
        ap.error("--dump-outputs writes the table of the count workload of --impl b200")
    global K, METRIC
    if args.config == "c3":
        args.k = 31
    K = args.k
    METRIC = f"kmers_counted_per_sec_k{K}"
    if args.warmup < 3 and args.impl == "b200":
        print(f"note: warmup {args.warmup} < 3 is below the timing rule", file=sys.stderr)
    if args.impl == "reference":
        return run_reference(args)
    if args.workload != "count":
        return run_secondary(args)

    import torch
    import torch.distributed as dist
    g, api, datagen = load_pkg()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if args.gpus > 1:
            raise SystemExit(f"--gpus {args.gpus} needs torchrun with {args.gpus} ranks (WORLD_SIZE={world})")
    torch.cuda.set_device(local_rank)
    # before any pinned allocation: run (and allocate) on the NUMA node the GPU hangs off
    from kmer_extension_b200 import hostbind
    placement = hostbind.bind_to_gpu(local_rank) if not os.environ.get("KMER_NO_BIND") else {"bound": False, "why": "KMER_NO_BIND"}
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    eng = api.KmerCuda(local_rank)
    n_rows = args.reads
    scaling = "weak"
    if args.config in ("c3", "c2x10"):                  # 10 GB in total, split by row over the ranks
        n_rows = 10_000_000 // world
        scaling = "strong"
    seed = 3 if args.config == "c3" else 2
    if args.devgen:
        # rows [rank*n_rows, (rank+1)*n_rows) of ONE seeded table, generated in HBM (csrc/synth.cu); the host copy is only what
        # the e2e arm and the oracle's checksum read
        nb = n_rows * READ_LEN
        g_seq = torch.zeros(((nb + 15) & ~15) + 64, dtype=torch.uint8, device="cuda")
        g_off = torch.zeros(n_rows + 1, dtype=torch.int64, device="cuda")
        eng.dev_synth_reads(seed, rank * n_rows, n_rows, READ_LEN, g_seq, g_off)
        eng.dev_finish()
        flat = g_seq[:nb].cpu().numpy()
        off = g_off.cpu().numpy().astype(np.uint64)
        del g_seq, g_off
    else:
        flat, off = datagen.synth_reads(seed + rank, n_rows, READ_LEN)
    n_bases = int(off[-1])
    n_kmers = n_rows * (READ_LEN - K + 1)          # per GPU (weak scaling: every rank brings its own 1 GB)
    total_kmers = n_kmers * world

    # ---------------------------------------------------------------- resident-data arm
    h_seq = torch.empty(n_bases + 64, dtype=torch.uint8).pin_memory()
    h_seq[:n_bases] = torch.from_numpy(flat)
    h_seq[n_bases:] = 0
    h_off = torch.from_numpy(off.astype(np.int64)).pin_memory()
    d_seq = h_seq.cuda(non_blocking=True)
    d_off = h_off.cuda(non_blocking=True)
    cap = eng.max_kmers(n_bases, n_rows, K)
    if world > 1:
        cap = int(cap * 1.1) + (1 << 20)              # an owner's share of the groups fluctuates a little
    d_pairs = torch.empty((cap, 2), dtype=torch.int64, device="cuda")
    stream = torch.cuda.current_stream()
    torch.cuda.synchronize()
    sharder = None
    if world > 1:
        from kmer_extension_b200 import sharded
        sharder = sharded.ShardedCounter(eng)

    class _R:
        pass

    def step():
        if sharder is None:
            eng.dev_count(d_seq, n_bases, d_off, n_rows, K, d_pairs, algo=args.algo, stream=stream)
            return eng.dev_finish(stream)
        nd, nk, info = sharder.count(d_seq, n_bases, d_off, n_rows, K, d_pairs, total_kmers=total_kmers)
        r = _R()
        r.n_kmers, r.n_distinct, r.n_overflow, r.n_tier2 = nk, nd, 0, info["tier2_kmers"]
        return r

    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        res = step()
    if world == 1:
        assert res.n_kmers == n_kmers, (res.n_kmers, n_kmers)
    n_distinct = int(res.n_distinct)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    barrier()
    sampler.mark_begin()
    l0 = eng.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        res = step()
    ev1.record(stream)
    barrier()
    sampler.mark_end()
    launches = eng.launches - l0
    clocks = sampler.stop()
    ms_total = ev0.elapsed_time(ev1)
    if world > 1:                                      # device time, max over ranks
        tmax = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms_total = float(tmax.item())
        dsum = torch.tensor([n_distinct], dtype=torch.int64, device="cuda")
        dist.all_reduce(dsum)
        n_distinct_total = int(dsum.item())
    else:
        n_distinct_total = n_distinct
    ms_step = ms_total / args.steps
    value = total_kmers * args.steps / (ms_total * 1e-3)
    if args.dump_outputs:                              # every rank holds its own share of the groups when world > 1
        dump_count_table(torch, args.dump_outputs, d_pairs[:int(res.n_distinct)], int(res.n_kmers),
                         suffix=f"_rank{rank}" if world > 1 else "", sample=(1 << 20) // world)

    # ---------------------------------------------------------------- parity of the table the LAST timed step left in HBM
    parity = {"what": "sum(count*mix64(code)) over the table == sum(mix64(code)) over all windows of the input rows (C oracle), "
                      "sum(count) == windows, keys unique (device sort); N>1: sums all-reduced, keys re-partitioned by hash "
                      "across ranks and checked unique there"}
    if not args.no_parity:
        nd_last = int(res.n_distinct)
        t_in = time.perf_counter()
        in_sum, in_n = input_checksum(flat, off, K)
        parity["oracle_seconds"] = time.perf_counter() - t_in
        keys_t, counts_t = d_pairs[:nd_last, 0], d_pairs[:nd_last, 1]
        tab_sum, tab_cnt = table_checksum(torch, keys_t, counts_t)
        uniq_ok = keys_unique(torch, keys_t)
        if world > 1:
            v = torch.tensor([_s64(in_sum), in_n, _s64(tab_sum), tab_cnt, 0 if uniq_ok else 1], dtype=torch.int64, device="cuda")
            dist.all_reduce(v)
            in_sum, in_n, tab_sum, tab_cnt = int(v[0].item()) & M64, int(v[1].item()), int(v[2].item()) & M64, int(v[3].item())
            uniq_ok = int(v[4].item()) == 0
            # a group split over two owners keeps both sums: send every key to rank hash(key) % world and look for duplicates there
            dest = ((mix64_torch(torch, keys_t) >> 17) & 0xffff) % world
            order = torch.argsort(dest)
            send = keys_t[order].contiguous()
            scnt = torch.bincount(dest, minlength=world)
            rcnt = torch.empty_like(scnt)
            dist.all_to_all_single(rcnt, scnt)
            recv = torch.empty(int(rcnt.sum().item()), dtype=torch.int64, device="cuda")
            dist.all_to_all_single(recv, send, output_split_sizes=rcnt.tolist(), input_split_sizes=scnt.tolist())
            cross = torch.tensor([0 if keys_unique(torch, recv) else 1], dtype=torch.int64, device="cuda")
            dist.all_reduce(cross)
            parity["cross_rank_unique_ok"] = int(cross.item()) == 0
            uniq_ok = uniq_ok and parity["cross_rank_unique_ok"]
            del dest, order, send, recv
        parity.update({"checksum_ok": in_sum == tab_sum, "count_ok": in_n == tab_cnt == total_kmers, "unique_ok": bool(uniq_ok),
                       "windows": in_n, "groups_checked_rank0": nd_last})
        torch.cuda.empty_cache()
    else:
        parity["skipped"] = True

    # ---------------------------------------------------------------- per-kernel phases (separate pass, not the timed one)
    eng.set_profiling(True)
    phase_acc = {}
    for _ in range(max(2, min(args.steps, 5))):
        step()
        for name, ms in (sharder.last_phases if sharder is not None else eng.phases()):
            phase_acc.setdefault(name, []).append(ms)
    eng.set_profiling(False)
    phases = {n: float(np.mean(v)) for n, v in phase_acc.items()}
    peak, peak_src = measured_peaks()
    b_alg_step = n_bases * world + 16 * n_distinct_total
    # algorithmic bytes of each kernel (DESIGN.md "Kernels"): what it must read + write once
    alg_bytes = {
        "count_hash_insert": n_bases + 16 * n_distinct,          # read every base once, create every group once
        "hash_compact": 16 * n_distinct * 2,                     # read + write every group once
        "hash_clear": 0,
        "count_dense+compact": n_bases + 16 * n_distinct,
        "minimizer_partition": n_bases,                         # compulsory: read every base once (records are overhead)
        "bucket_count": 16 * n_distinct,                        # compulsory: write every group once
        "tier2_insert": 0, "tier2_compact": 0,
    }
    # DRAM traffic per launch from the committed `ncu --set full` capture of this workload (profiles/), if there is one
    traffic = {}
    tp = ROOT / "profiles" / "r02_dram_traffic_1g_k21.json"
    if tp.exists() and world == 1 and n_rows == 1_000_000:
        try:
            traffic = json.loads(tp.read_text())["kernels"]
        except Exception:
            traffic = {}

    def kernel_roofline(name):
        ab = alg_bytes.get(name, b_alg_step)
        ach = ab / (phases[name] * 1e-3) / 1e9
        return {"bound": "hbm", "kernel": name, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": traffic.get(name), "alg_bytes_per_launch": ab, "kernel_ms": phases[name],
                "share_of_step": phases[name] / max(sum(phases.values()), 1e-9), "peak_source": peak_src}

    dom = max(phases, key=phases.get) if phases else None
    roofline = kernel_roofline(dom) if dom else None
    # the two kernels of the count take the same time to within a few per cent: both are listed, whichever leads
    roofline_kernels = [kernel_roofline(n) for n in sorted(phases, key=phases.get, reverse=True)[:2]] if phases else []
    ach_step = b_alg_step / (ms_step * 1e-3) / 1e9
    roofline_step = {"bound": "hbm", "achieved": ach_step, "peak": peak * world, "unit": "GB/s", "frac": ach_step / (peak * world),
                     "alg_bytes_per_step": b_alg_step, "formula": "N_bases + 16*D over all GPUs (SURVEY 8d); peak = n_gpus x measured HBM copy",
                     "frac_of_8000_nominal": ach_step / (8000.0 * world)}

    # ---------------------------------------------------------------- e2e arm: host buffers through the C ABI
    e2e = None
    if not args.no_e2e:
        import psutil
        need = 16 * n_distinct + (1 << 30)
        if psutil.virtual_memory().available < 2 * need * max(world, 1):
            e2e = {"value": None, "unit": UNIT, "skipped": "host memory too small for a pinned result buffer"}
        elif world == 1:
            pairs, d, nk = C.c_void_p(), C.c_uint64(), C.c_uint64()
            uq, nu = C.c_void_p(), C.c_uint64()
            seq_ptr, off_ptr = h_seq.data_ptr(), h_off.data_ptr()

            in_chk = input_checksum(flat, off, K) if not args.no_parity else None

            def host_view(ptr, n_items, dtype):
                return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), shape=(n_items * np.dtype(dtype).itemsize,)).view(dtype)

            def check_table(uniq_codes, pair_arr):
                """the host result of one e2e call (unique codes as int64 array or None, pairs as [n,2] int64) against the oracle's checksum"""
                tot, cnt, ok_u = 0, 0, True
                allkeys = []
                if uniq_codes is not None and uniq_codes.size:
                    ku = torch.from_numpy(uniq_codes).cuda()
                    a, b = table_checksum(torch, ku)
                    tot, cnt = (tot + a) & M64, cnt + b
                    allkeys.append(ku)
                if pair_arr.size:
                    pa = torch.from_numpy(pair_arr).cuda()
                    a, b = table_checksum(torch, pa[:, 0], pa[:, 1])
                    tot, cnt = (tot + a) & M64, cnt + b
                    allkeys.append(pa[:, 0].contiguous())
                    del pa
                ok_u = keys_unique(torch, torch.cat(allkeys)) if allkeys else True
                del allkeys
                torch.cuda.empty_cache()
                return {"checksum_ok": tot == in_chk[0], "count_ok": cnt == in_chk[1], "unique_ok": ok_u}

            def e2e_step_pairs(check=False):
                rc = eng.lib.kmer_cuda_submit_count(eng.ctx, seq_ptr, off_ptr, n_rows, K, C.byref(pairs), C.byref(d), C.byref(nk))
                if rc:
                    eng._raise(eng.ctx)
                chk = (C.c_uint64 * 2).from_address(pairs.value)  # touch the result on the host
                got = [int(chk[0]), int(chk[1]), int(d.value), int(nk.value), 16 * int(d.value), None]
                if check:
                    got[5] = check_table(None, host_view(pairs, 2 * int(d.value), np.int64).reshape(-1, 2))
                eng.lib.kmer_cuda_release(eng.ctx, pairs)
                return got

            def e2e_step_split(check=False):
                rc = eng.lib.kmer_cuda_submit_count_split(eng.ctx, seq_ptr, off_ptr, n_rows, K, C.byref(uq), C.byref(nu),
                                                          C.byref(pairs), C.byref(d), C.byref(nk))
                if rc:
                    eng._raise(eng.ctx)
                chk = (C.c_uint64 * 1).from_address(uq.value) if nu.value else [0]  # touch the result on the host
                got = [int(chk[0]), 0, int(d.value) + int(nu.value), int(nk.value), 16 * int(d.value) + 8 * int(nu.value), None]
                if check:
                    got[5] = check_table(host_view(uq, int(nu.value), np.int64), host_view(pairs, 2 * int(d.value), np.int64).reshape(-1, 2))
                eng.lib.kmer_cuda_release(eng.ctx, uq)
                eng.lib.kmer_cuda_release(eng.ctx, pairs)
                return got

            nbytes_c = C.c_int()

            def e2e_step_packed(check=False):
                rc = eng.lib.kmer_cuda_submit_count_packed(eng.ctx, seq_ptr, off_ptr, n_rows, K, C.byref(uq), C.byref(nu), C.byref(nbytes_c),
                                                           C.byref(pairs), C.byref(d), C.byref(nk))
                if rc:
                    eng._raise(eng.ctx)
                chk = (C.c_uint8 * 8).from_address(uq.value) if nu.value else [0]  # touch the result on the host
                got = [int(chk[0]), 0, int(d.value) + int(nu.value), int(nk.value), 16 * int(d.value) + nbytes_c.value * int(nu.value), None]
                if check:
                    nb = nbytes_c.value
                    raw = torch.from_numpy(host_view(uq, int(nu.value) * nb, np.uint8)).cuda().view(-1, nb).to(torch.int64)
                    codes = torch.zeros(raw.shape[0], dtype=torch.int64, device="cuda")
                    for j in range(nb):                         # little-endian ceil(2k/8)-byte integers
                        codes |= raw[:, j] << (8 * j)
                    del raw
                    got[5] = check_table(codes.cpu().numpy(), host_view(pairs, 2 * int(d.value), np.int64).reshape(-1, 2))
                eng.lib.kmer_cuda_release(eng.ctx, uq)
                eng.lib.kmer_cuda_release(eng.ctx, pairs)
                return got

            def timed(step_fn, api_name):
                e2e_steps = max(1, min(args.steps, 3))
                for _ in range(2):
                    step_fn()
                t0 = time.perf_counter()
                for _ in range(e2e_steps):
                    got = step_fn()
                dt = time.perf_counter() - t0
                assert got[2] == n_distinct and got[3] == n_kmers
                r = {"value": n_kmers * e2e_steps / dt, "unit": UNIT, "h2d_bytes_per_step": n_bases + 8 * (n_rows + 1),
                     "d2h_bytes_per_step": got[4], "ms_per_step": 1e3 * dt / e2e_steps, "steps": e2e_steps, "api": api_name}
                if not args.no_parity:                           # one more call, untimed, whose host result is checked
                    r["parity"] = step_fn(check=True)[5]
                return r

            # the result of the GROUP BY crosses PCIe either as 16-byte (k-mer, count) pairs, or in the split format
            # (a group with count 1 as its bare 8-byte code, the rest as pairs): same table, half the bytes on this input
            e2e = timed(e2e_step_packed, "kmer_cuda_submit_count_packed (pinned host input -> pinned host result: unique k-mers as "
                                         "bare ceil(2k/8)-byte codes + (k-mer,count) pairs for the rest)")
            e2e["split_format"] = timed(e2e_step_split, "kmer_cuda_submit_count_split (unique k-mers as bare 8-byte codes + pairs)")
            e2e["pairs_format"] = timed(e2e_step_pairs, "kmer_cuda_submit_count (pinned host input -> pinned host (k-mer,count) table)")
            # what the PostgreSQL glue feeds: palloc'ed, i.e. PAGEABLE, input (the driver stages it through its own pinned buffers)
            pg_seq = np.ascontiguousarray(flat)
            pg_off = np.ascontiguousarray(off.astype(np.uint64))
            seq_ptr, off_ptr = pg_seq.ctypes.data, pg_off.ctypes.data
            e2e["pageable_input"] = timed(e2e_step_packed, "kmer_cuda_submit_count_packed with PAGEABLE host input (what palloc gives the glue)")
            seq_ptr, off_ptr = h_seq.data_ptr(), h_off.data_ptr()
        else:
            # sharded e2e: every rank copies its rows from pinned host memory, counts with the all-to-all, and reads
            # its share of the (k-mer,count) table back into pinned host memory
            # (split result format: groups with count 1 as bare 8-byte codes, the rest as 16-byte pairs)
            nbytes = (2 * K + 7) // 8                       # bare codes cross PCIe as ceil(2k/8)-byte integers (6 at k=21)
            h_pairs = torch.empty((cap // 2 + (1 << 20), 2), dtype=torch.int64).pin_memory()
            h_packed = torch.empty(cap * nbytes + 16, dtype=torch.uint8).pin_memory()
            d_uniq = torch.empty(cap, dtype=torch.int64, device="cuda")
            d_packed = torch.empty(cap * nbytes + 16, dtype=torch.uint8, device="cuda")
            d2h_bytes = [0]
            e2e_last = [0, 0]
            ev_d2h = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            d2h_ms = [0.0]

            def e2e_step():
                d_seq.copy_(h_seq, non_blocking=True)
                d_off.copy_(h_off, non_blocking=True)
                nd, nk_, info = sharder.count(d_seq, n_bases, d_off, n_rows, K, d_pairs, total_kmers=total_kmers, d_uniq=d_uniq)
                nu = info["n_unique"]
                ev_d2h[0].record()
                h_pairs[:nd].copy_(d_pairs[:nd], non_blocking=True)
                ev_d2h[1].record()
                eng.dev_pack_codes(d_uniq, nu, K, d_packed, stream=stream)
                h_packed[:nu * nbytes].copy_(d_packed[:nu * nbytes], non_blocking=True)
                ev_d2h[2].record()
                torch.cuda.synchronize()
                d2h_ms[0] = ev_d2h[0].elapsed_time(ev_d2h[2])     # both copies + the pack kernel between them
                d2h_bytes[0] = 16 * nd + nbytes * nu
                e2e_last[0], e2e_last[1] = nd, nu
                return nd + nu, int(h_packed[0]) if nu else 0

            e2e_steps = max(1, min(args.steps, 3))
            for _ in range(2):
                e2e_step()
            barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                nd, _ = e2e_step()
            barrier()
            dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            dt = float(dt.item())
            d2h_sum = torch.tensor([d2h_bytes[0]], dtype=torch.int64, device="cuda")
            dist.all_reduce(d2h_sum)
            # per-rank D2H rate of the last step (device events around the result copies) and where each rank's host side runs
            mine = torch.tensor([d2h_bytes[0] / max(d2h_ms[0], 1e-6) / 1e6, float(placement.get("numa_node") if placement.get("numa_node") is not None else -1),
                                 1.0 if placement.get("bound") else 0.0], dtype=torch.float64, device="cuda")
            per_rank = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(per_rank, mine)
            e2e_parity = None
            if not args.no_parity:                               # the HOST copies of the last step against the oracle's checksum
                nd_h, nu_h = int(e2e_last[0]), int(e2e_last[1])
                raw = h_packed[:nu_h * nbytes].cuda().view(-1, nbytes).to(torch.int64)
                codes_h = torch.zeros(nu_h, dtype=torch.int64, device="cuda")
                for j in range(nbytes):
                    codes_h |= raw[:, j] << (8 * j)
                del raw
                a1, c1 = table_checksum(torch, codes_h)
                del codes_h
                hp = h_pairs[:nd_h].cuda()
                a2, c2 = table_checksum(torch, hp[:, 0], hp[:, 1]) if nd_h else (0, 0)
                in_sum2, in_n2 = input_checksum(flat, off, K)
                v = torch.tensor([_s64(in_sum2), in_n2, _s64((a1 + a2) & M64), c1 + c2], dtype=torch.int64, device="cuda")
                dist.all_reduce(v)
                e2e_parity = {"checksum_ok": (int(v[0].item()) & M64) == (int(v[2].item()) & M64), "count_ok": int(v[1].item()) == int(v[3].item())}
                del hp
            e2e = {"value": total_kmers * e2e_steps / dt, "unit": UNIT, "h2d_bytes_per_step": (n_bases + 8 * (n_rows + 1)) * world,
                   "d2h_bytes_per_step": int(d2h_sum.item()), "ms_per_step": 1e3 * dt / e2e_steps, "steps": e2e_steps,
                   "api": "ShardedCounter.count per rank: pinned host rows -> HBM, partition + split (pulls the peers' segments over NVLink) + bucket count, "
                          "this rank's share of the table (packed split format: ceil(2k/8)-byte codes + pairs) -> pinned host",
                   "d2h_gb_per_s_per_rank_mean": float(d2h_sum.item()) / world / max(dt / e2e_steps, 1e-9) / 1e9,
                   "d2h_copy_gb_per_s_per_rank": [round(float(x[0].item()), 2) for x in per_rank],
                   "host_numa_node_per_rank": [int(x[1].item()) for x in per_rank],
                   "host_bound_to_gpu_node_per_rank": [bool(x[2].item()) for x in per_rank],
                   "parity": e2e_parity}

    # ---------------------------------------------------------------- CPU baseline beside it (rank 0, bounded sample)
    cpu = None
    if not args.no_cpu and rank == 0:
        try:
            r = cpu_reference_run(datagen, args.cpu_reads, host_threads(), 1, 0)
            cpu = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
        except Exception as ex:  # the baseline must never take the GPU number down with it
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {ex}"}

    # ---------------------------------------------------------------- the other rows of the path, short (rank 0, N=1 only)
    secondary = None
    if world == 1 and not args.no_secondary:
        secondary = {}
        del d_pairs
        torch.cuda.empty_cache()

        def timed_dev(fn, reps=5):
            for _ in range(2):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(reps):
                fn()
            e1.record(stream)
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / reps

        def sec_line(what, ms, alg, units, unit):
            ach = alg / (ms * 1e-3) / 1e9
            return {"workload": what, "ms": ms, "value": units / (ms * 1e-3), "unit": unit,
                    "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "alg_bytes": alg}}

        try:
            # generate_kmers over the resident column: B_alg = N + 8 * n_kmers
            d_codes = torch.empty(n_kmers, dtype=torch.int64, device="cuda")

            def f_extract():
                eng.dev_extract(d_seq, n_bases, d_off, n_rows, K, d_codes, stream=stream)
                eng.dev_finish(stream)
            secondary["extract"] = sec_line(f"generate_kmers over {n_bases / 1e9:.3g} GB, k={K}", timed_dev(f_extract), n_bases + 8 * n_kmers,
                                            n_kmers, "k-mers/s")
            del d_codes
            torch.cuda.empty_cache()
            # configs[4] at a quarter of its size: equals + starts_with in ONE pass over M 32-mers: B_alg = 8 M + 2 M/8
            m5 = 250_000_000
            g = torch.Generator(device="cuda").manual_seed(5)
            col5 = (torch.randint(0, 1 << 32, (m5,), dtype=torch.int64, device="cuda", generator=g) << 32) | \
                torch.randint(0, 1 << 32, (m5,), dtype=torch.int64, device="cuda", generator=g)   # uniform 32-mers
            c0 = int(col5[0].item()) & M64
            txt = "".join("acgt"[(c0 >> (2 * (31 - j))) & 3] for j in range(32))
            bits5 = torch.empty(2 * ((m5 + 31) // 32), dtype=torch.int32, device="cuda")
            hits5 = torch.empty(2, dtype=torch.int64, device="cuda")

            def f_c5():
                eng.dev_match(api.OP_EQUALS, col5, m5, 32, [txt, txt[:8]], bits5, hits5, ops=[api.OP_EQUALS, api.OP_STARTS_WITH], stream=stream)
                eng.dev_finish(stream)
            secondary["match_c5"] = sec_line(f"configs[4] at 1/4 size: equals + starts_with(8-base prefix) in one pass over {m5:.3g} 32-mers",
                                             timed_dev(f_c5), 8 * m5 + 2 * ((m5 + 7) // 8), 2 * m5, "pair-tests/s")
            del col5, bits5, hits5
            torch.cuda.empty_cache()
            # configs[3] at a quarter of its size: contains, 1000 IUPAC patterns (k=12) x M k-mers, full bit matrix
            m4, P = 25_000_000, 1000
            col4 = torch.randint(0, 1 << 24, (m4,), dtype=torch.int64, device="cuda", generator=g)
            pats = datagen.synth_qkmers(4, P, 12, with_n=True)
            bits4 = torch.empty(P * ((m4 + 31) // 32), dtype=torch.int32, device="cuda")
            hits4 = torch.empty(P, dtype=torch.int64, device="cuda")

            def f_c4():
                eng.dev_match(api.OP_CONTAINS, col4, m4, 12, pats, bits4, hits4, stream=stream)
                eng.dev_finish(stream)
            ms4 = timed_dev(f_c4, reps=3)
            secondary["match_c4"] = sec_line(f"configs[3] at 1/4 size: contains, {P} IUPAC patterns (k=12) x {m4:.3g} k-mers, full bit matrix",
                                             ms4, 8 * m4 + 16 * P + P * ((m4 + 7) // 8), m4 * P, "pair-tests/s")
            # SURVEY 8d3: this kernel is INT32-bound, not HBM-bound -- its fraction of the integer issue rates, from the static SASS
            # count of its round loop (tools/sass_loop_count.py -> profiles/), the trip count of this workload and the measured time
            sp = ROOT / "profiles" / "r02_match_table_sass_counts.json"
            if sp.exists():
                sc = json.loads(sp.read_text())
                trips = ((m4 + 31) // 32) * ((P + 1023) // 1024)                 # warp rounds: 32 k-mers x one group of 1024 constants
                mhz = clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965.0
                sm_count = torch.cuda.get_device_properties(0).multi_processor_count
                smsp_cycles = ms4 * 1e-3 * mhz * 1e6 * sm_count * 4               # cycles x SM sub-partitions
                alu, allins = sc["by_pipe"].get("alu", 0), sc["instructions"]
                secondary["match_c4"]["int32"] = {
                    "alu_pipe_frac": trips * alu * 2.0 / smsp_cycles,             # LOP3/SHF/...: one warp instruction per 2 cycles per sub-partition
                    "issue_slot_frac": trips * allins / smsp_cycles,              # any instruction: one per cycle per sub-partition
                    "warp_instr_per_round": allins, "alu_pipe_warp_instr_per_round": alu, "rounds": trips,
                    "pair_tests_per_round": sc["pair_tests_per_loop_trip"], "sm_mhz": mhz, "sm_count": sm_count,
                    "source": "static SASS count of the round loop (profiles/r02_match_table_sass_counts.json) x trip count / measured time; "
                              "pipe rates from B300_MICROARCH.md (alu pipe rt_SMSP = 2); an estimate, not an ncu counter"}
            del col4, bits4, hits4
            torch.cuda.empty_cache()
        except Exception as ex:                            # the secondary rows must never take the headline down
            secondary["error"] = repr(ex)

    # SURVEY 8d3: multi-GPU runs also state their NVLink traffic against 900 GB/s per direction per GPU
    nvlink = None
    try:
        if sharder is not None:
            pulled = sharder._pull is not None
            ms_x = phases.get("refine") if pulled else phases.get("exchange")
            if ms_x:
                xb = int(sharder.last_exchange_bytes)      # pull: filled records + fill words of this rank's send block that OTHER owners read
                gbs = xb / (ms_x * 1e-3) / 1e9
                nvlink = {"bytes_per_gpu_per_step": xb,
                          "kernel": ("refine (the owner's split kernel pulls its segments from the peers' HBM; the transfer overlaps its own work)"
                                     if pulled else "exchange (NCCL all_to_all of the segments, capacity not fill)"),
                          "kernel_ms": ms_x, "gb_per_s_per_direction": gbs, "peak": 900.0, "frac": gbs / 900.0,
                          "what": "rank 0's egress = what its peers take out of its send block, by symmetry each GPU's ingress; counted from "
                                  "the fill words / buffer sizes, not a hardware counter"}
    except Exception as ex:                               # never take the headline down
        nvlink = {"error": repr(ex)}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "u64",
            "data": "synthetic",
            "config": {"workload": workload_name(args.config, K, n_rows),
                       "k": K, "read_len": READ_LEN,
                       "reads_per_gpu": n_rows, "algo": args.algo, "n_kmers_per_step": n_kmers * world,
                       "n_distinct_rank0": n_distinct, "recounted_kmers": int(res.n_overflow),
                       "tier2_kmers": int(res.n_tier2), "n_distinct_total": n_distinct_total,
                       "exchange_bytes_per_gpu_per_step": (sharder.last_exchange_bytes if sharder is not None else 0),
                       "exchange": (None if sharder is None else ("peer reads inside the split kernel (CUDA IPC over NVLink)" if sharder._pull is not None
                                                                  else "NCCL all_to_all")),
                       "generator": ("device: counter-based table, csrc/synth.cu, rows split over the ranks" if args.devgen
                                     else "host: numpy PCG64, seed + rank"),
                       "host_placement_rank0": placement, "l2": "inputs and tables larger than L2 (no flush needed)",
                       "bases_per_sec": n_bases * world * args.steps / (ms_total * 1e-3)},
            "roofline": roofline, "roofline_kernels": roofline_kernels, "roofline_step": roofline_step, "phases_ms": phases, "cpu_baseline": cpu, "e2e": e2e,
            "parity": parity, "secondary": secondary, "nvlink": nvlink, "gpu_launches": int(launches), "clocks": clocks}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if sharder is not None:
        sharder.close()
    eng.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    bad = [k for k in ("checksum_ok", "count_ok", "unique_ok") if parity.get(k) is False]
    for fmt in ([e2e] + [e2e.get("split_format"), e2e.get("pairs_format")] if isinstance(e2e, dict) else []):
        if isinstance(fmt, dict) and isinstance(fmt.get("parity"), dict):
            bad += [f"e2e:{k}" for k, v in fmt["parity"].items() if v is False]
    if bad:
        raise SystemExit(f"PARITY FAILURE: {bad}")


if __name__ == "__main__":
    main()
