"""Cost of canonical counting against the strand-specific count, on one GPU; prints one JSON line.

In one process, alternating step by step on the same seeded inputs:
  * resident ms/step of kmer_cuda_dev_count and kmer_cuda_dev_count_canonical (pairs in HBM), with the per-kernel phases of one
    profiled call of each (kmer_cuda_get_phases), and the tier-2 share (n_tier2 / n_kmers) and recount flag of each;
  * end to end from host buffers: kmer_cuda_submit_count and kmer_cuda_submit_count_canonical (pairs), each call blocking until
    its table is in pinned host memory.
Workloads: the bench workload (1e6 uniform reads x 1000 bases, seed 2, k = 21) and 256 MiB of 1000-base reads of one genome at
30x coverage with 0.2 % substitutions, every other read reverse-complemented (reads from both strands; tests/coverage_util.py,
tests/canonical_util.py).  The GPU's name and power limit are read in the same run.

    python tools/canonical_bench.py --steps 10 --warmup 2
"""
import argparse
import ctypes as C
import json
import statistics
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
sys.path.insert(0, str(ROOT / "tools"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--k", type=int, default=21)
    a = ap.parse_args()
    import torch
    import __graft_entry__ as g
    g.load_package()
    import canonical_util as CN
    import coverage_util as CU
    from kmer_extension_b200 import api, datagen
    from spectrum_bench import gpu_info

    if not torch.cuda.is_available():
        raise SystemExit("canonical_bench: no CUDA device (there is no CPU measurement)")
    eng = api.KmerCuda(0)
    lib, k = eng.lib, a.k
    inputs = {"uniform_seed2": datagen.synth_reads(2, 1_000_000, 1000)}
    n_reads = (256 << 20) // 1000
    (flat, off), _ = CU.sample_reads(11, n_reads * 1000 // 30, n_reads, 1000, 0.002)
    inputs["coverage30x_both_strands_256MiB"] = (CN.revcomp_rows(flat, off, np.arange(n_reads) % 2 == 1), off)
    result = {"tool": "canonical_bench", "gpu": gpu_info(), "k": k, "steps": a.steps, "workloads": {}}

    for name, (flat, off) in inputs.items():
        off = np.asarray(off, np.uint64)
        n_bases, n_rows = int(off[-1]), len(off) - 1
        n = eng.max_kmers(n_bases, n_rows, k)
        d_seq = torch.from_numpy(np.concatenate([flat, np.zeros(80, np.uint8)])).cuda()
        d_off = torch.from_numpy(off.view(np.int64).copy()).cuda()
        pairs = torch.empty((n, 2), dtype=torch.int64, device="cuda")

        def run(canonical):
            eng.dev_count(d_seq, n_bases, d_off, n_rows, k, pairs, canonical=canonical)
            return eng.dev_finish()

        def timed(canonical):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            r = run(canonical)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1), r

        for _ in range(a.warmup):
            run(False)
            run(True)
        t = {False: [], True: []}
        res = {}
        for _ in range(a.steps):                  # alternating
            for cn in (False, True):
                ms, res[cn] = timed(cn)
                t[cn].append(ms)
        phases = {}
        eng.set_profiling(True)
        for cn in (False, True):
            run(cn)
            phases["canonical" if cn else "strand_specific"] = [(p, round(ms, 3)) for p, ms in eng.phases()]
        eng.set_profiling(False)
        del pairs
        torch.cuda.empty_cache()
        fl = np.ascontiguousarray(flat)
        e2e = {False: [], True: []}
        for i in range(a.e2e_steps + 1):
            for cn in (False, True):
                pp, npairs, nk = C.c_void_p(), C.c_uint64(), C.c_uint64()
                t0 = time.perf_counter()
                if cn:
                    eng._check(lib.kmer_cuda_submit_count_canonical(eng.ctx, fl.ctypes.data, off.ctypes.data, n_rows, k, None, None,
                                                                    C.byref(pp), C.byref(npairs), C.byref(nk)))
                else:
                    eng._check(lib.kmer_cuda_submit_count(eng.ctx, fl.ctypes.data, off.ctypes.data, n_rows, k, C.byref(pp),
                                                          C.byref(npairs), C.byref(nk)))
                t1 = time.perf_counter()
                lib.kmer_cuda_release(eng.ctx, pp)
                if i:                              # the first pair warms the pinned pools
                    e2e[cn].append((t1 - t0) * 1e3)
        med = statistics.median
        w = {}
        for cn in (False, True):
            r = res[cn]
            w["canonical" if cn else "strand_specific"] = {
                "groups": int(r.n_distinct), "n_kmers": int(r.n_kmers), "tier2_share": round(r.n_tier2 / max(r.n_kmers, 1), 5),
                "recounted": bool(r.n_overflow), "resident_ms": round(med(t[cn]), 3), "resident_ms_all": [round(x, 3) for x in t[cn]],
                "e2e_ms": round(med(e2e[cn]), 1), "e2e_ms_all": [round(x, 1) for x in e2e[cn]]}
        w["resident_ratio"] = round(w["canonical"]["resident_ms"] / w["strand_specific"]["resident_ms"], 4)
        w["e2e_ratio"] = round(w["canonical"]["e2e_ms"] / w["strand_specific"]["e2e_ms"], 4)
        w["phases_ms"] = phases
        result["workloads"][name] = w
        del d_seq, d_off
        torch.cuda.empty_cache()
    eng.close()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
