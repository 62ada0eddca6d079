"""Resident and end-to-end cost of the abundance spectrum against the GROUP BY it summarises, on one GPU; prints one JSON line.

In one process, alternating step by step on the same inputs:
  * resident ms/step of kmer_cuda_dev_count (the (code, count) table in HBM) and kmer_cuda_dev_count_spectrum (hist + tail),
    with the per-kernel phases of one profiled call of each (kmer_cuda_get_phases);
  * end to end from host buffers: kmer_cuda_submit_count_packed (the table across PCIe, its smallest format) and
    kmer_cuda_submit_count_spectrum;
  * parity in the same run: dev_pairs_spectrum(dev_count's table) == dev_count_spectrum, and sum c * hist[c] + tail = windows.
Workloads: the bench workload (1e6 uniform reads x 1000 bases, seed 2, k = 21) and 1e6 reads x 1000 of one genome at 10x
coverage with 0.2 % substitutions (tests/coverage_util.py, seed 11).  The GPU's name and power limit are read in the same run.

    python tools/spectrum_bench.py --steps 10 --warmup 2
"""
import argparse
import ctypes as C
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.splitlines()[0]
        name, power, clk = (x.strip() for x in out.split(","))
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:                       # noqa: BLE001
        return {"name": None, "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--hist-len", type=int, default=65536)
    ap.add_argument("--k", type=int, default=21)
    a = ap.parse_args()
    import torch
    import __graft_entry__ as g
    g.load_package()
    import coverage_util as CU
    from kmer_extension_b200 import api, datagen

    if not torch.cuda.is_available():
        raise SystemExit("spectrum_bench: no CUDA device (there is no CPU measurement)")
    eng = api.KmerCuda(0)
    lib, k, H = eng.lib, a.k, a.hist_len
    n_reads, L = 1_000_000, 1000
    inputs = {"uniform_seed2": datagen.synth_reads(2, n_reads, L)}
    (flat, off), _ = CU.sample_reads(11, n_reads * L // 10, n_reads, L, 0.002)
    inputs["coverage10x_err0.002"] = (flat, off)
    result = {"tool": "spectrum_bench", "gpu": gpu_info(), "k": k, "hist_len": H, "steps": a.steps, "workloads": {}}

    for name, (flat, off) in inputs.items():
        off = np.asarray(off, np.uint64)
        n_bases, n_rows = int(off[-1]), len(off) - 1
        n = eng.max_kmers(n_bases, n_rows, k)
        d_seq = torch.from_numpy(np.concatenate([flat, np.zeros(80, np.uint8)])).cuda()
        d_off = torch.from_numpy(off.view(np.int64).copy()).cuda()
        pairs = torch.empty((n, 2), dtype=torch.int64, device="cuda")
        hist = torch.empty(H, dtype=torch.int64, device="cuda")
        tail = torch.empty((max(n // H, 1), 2), dtype=torch.int64, device="cuda")
        hist2, tail2 = torch.empty_like(hist), torch.empty_like(tail)

        def run_count():
            eng.dev_count(d_seq, n_bases, d_off, n_rows, k, pairs)
            return eng.dev_finish()

        def run_spectrum():
            eng.dev_count_spectrum(d_seq, n_bases, d_off, n_rows, k, hist, tail)
            return eng.dev_finish()

        def timed(fn):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            r = fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1), r

        for _ in range(a.warmup):
            run_count()
            run_spectrum()
        t_count, t_spec = [], []
        for _ in range(a.steps):                  # alternating
            t, rc = timed(run_count)
            t_count.append(t)
            t, rs = timed(run_spectrum)
            t_spec.append(t)
        phases = {}
        eng.set_profiling(True)
        for what, fn in (("dev_count", run_count), ("dev_count_spectrum", run_spectrum)):
            fn()
            phases[what] = [(p, round(ms, 3)) for p, ms in eng.phases()]
        eng.set_profiling(False)
        # parity: the spectrum of the table == the spectrum binned in the counter, and the invariant
        rc = run_count()
        eng.dev_pairs_spectrum(pairs, rc.n_distinct, hist2, tail2)
        rp = eng.dev_finish()
        rs = run_spectrum()
        h1, h2 = hist.cpu().numpy(), hist2.cpu().numpy()
        t1 = np.sort(tail[:rs.n_distinct].cpu().numpy().view(np.uint64), axis=0)
        t2 = np.sort(tail2[:rp.n_distinct].cpu().numpy().view(np.uint64), axis=0)
        total = int((np.arange(H, dtype=np.int64) * h1).sum()) + int(t1[:, 1].sum())
        parity = bool(np.array_equal(h1, h2) and np.array_equal(t1, t2) and total == n == rs.n_kmers)
        del pairs
        torch.cuda.empty_cache()
        # end to end from host buffers (each call blocks until its result is in pinned host memory)
        fl = np.ascontiguousarray(flat)
        e2e = {"submit_count_packed": [], "submit_count_spectrum": []}
        for i in range(a.e2e_steps + 1):
            uq, nu, nb, pp, npairs, nk = C.c_void_p(), C.c_uint64(), C.c_int(), C.c_void_p(), C.c_uint64(), C.c_uint64()
            t0 = time.perf_counter()
            eng._check(lib.kmer_cuda_submit_count_packed(eng.ctx, fl.ctypes.data, off.ctypes.data, n_rows, k, C.byref(uq), C.byref(nu),
                                                         C.byref(nb), C.byref(pp), C.byref(npairs), C.byref(nk)))
            t1_ = time.perf_counter()
            lib.kmer_cuda_release(eng.ctx, uq)
            lib.kmer_cuda_release(eng.ctx, pp)
            hp, tp, nt = C.c_void_p(), C.c_void_p(), C.c_uint64()
            t2_ = time.perf_counter()
            eng._check(lib.kmer_cuda_submit_count_spectrum(eng.ctx, fl.ctypes.data, off.ctypes.data, n_rows, k, H, C.byref(hp), C.byref(tp),
                                                           C.byref(nt), C.byref(nk)))
            t3_ = time.perf_counter()
            lib.kmer_cuda_release(eng.ctx, hp)
            lib.kmer_cuda_release(eng.ctx, tp)
            if i:                                  # the first pair warms the pinned pools
                e2e["submit_count_packed"].append((t1_ - t0) * 1e3)
                e2e["submit_count_spectrum"].append((t3_ - t2_) * 1e3)
        med = statistics.median
        result["workloads"][name] = {
            "n_kmers": n, "n_tier2": int(rs.n_tier2), "n_overflow": int(rs.n_overflow), "groups": int(rc.n_distinct),
            "tail_groups": int(rs.n_distinct), "hist1": int(h1[1]),
            "resident_ms": {"dev_count": round(med(t_count), 3), "dev_count_spectrum": round(med(t_spec), 3),
                            "dev_count_all": [round(x, 3) for x in t_count], "dev_count_spectrum_all": [round(x, 3) for x in t_spec]},
            "phases_ms": phases,
            "e2e_ms": {kk: round(med(v), 1) for kk, v in e2e.items()},
            "e2e_ms_all": {kk: [round(x, 1) for x in v] for kk, v in e2e.items()},
            "parity": parity,
        }
        del d_seq, d_off, hist, tail, hist2, tail2
        torch.cuda.empty_cache()
    eng.close()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
