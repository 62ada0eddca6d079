"""CPU (gloo, world size 2) test of ShardedCounter.spectrum's host logic: the owners' spectra through the exchange (k >= 14) and
the dense path (k <= 13), the combine (one all-reduce of the histograms, an all-gather of the tails), and error agreement.  The
CUDA engine cannot run here: the numpy stand-in of tests/test_sharded_cpu.py, extended by the spectrum calls, plays it."""
import ctypes as C
import os
import socket
import sys
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

from test_sharded_cpu import StandInEngine, _Res  # noqa: E402

HIST_LEN = 4


def _bin(keys, counts, hist, tail):
    """the spectrum format of the library: hist overwritten, groups with count >= len(hist) appended to the tail"""
    h = hist.numpy()
    h[:] = 0
    small = counts < h.size
    np.add.at(h, counts[small].astype(np.int64), 1)
    t = tail.numpy().view(np.uint64)
    n = int((~small).sum())
    assert n <= t.shape[0]
    t[:n, 0], t[:n, 1] = keys[~small], counts[~small]
    return n


class SpectrumStandIn(StandInEngine):
    def dev_shard_count_spectrum(self, plan, src_recs, src_fill, d_hist, d_tail, stream=None):
        got = []
        for ra, fa in zip(src_recs, src_fill):
            recs = np.ctypeslib.as_array((C.c_uint64 * (plan.buckets_per_rank * plan.cap)).from_address(int(ra)))
            fill = np.ctypeslib.as_array((C.c_int64 * plan.buckets_per_rank).from_address(int(fa)))
            for b in range(plan.buckets_per_rank):
                got.append(recs[b * plan.cap:b * plan.cap + int(fill[b] & 0xFFFFFFFF)])
        allc = np.concatenate(got) if got else np.zeros(0, np.uint64)
        keys, counts = np.unique(allc, return_counts=True)
        n = _bin(keys, counts.astype(np.uint64), d_hist, d_tail)
        self._res = _Res(n_kmers=int(allc.size), n_distinct=n)

    def dev_pairs_spectrum(self, d_pairs, n, d_hist, d_tail, stream=None):
        p = d_pairs.numpy().view(np.uint64)[:n]
        nt = _bin(p[:, 0].copy(), p[:, 1].copy(), d_hist, d_tail)
        self._res = _Res(n_kmers=int(p[:, 1].sum()), n_distinct=nt)


def _rows(rank):
    from kmer_extension_b200 import datagen
    flat, off = datagen.synth_ragged(300 + rank, 50, 80, min_len=32, mixed_case=True)
    rep = flat[int(off[0]):int(off[1])]                    # the first read again on every rank: counts >= HIST_LEN
    flat = np.concatenate([flat, rep, rep, np.frombuffer(b"ACGT" * 20, np.uint8)])
    off = np.concatenate([off, off[-1] + np.cumsum([rep.size, rep.size, 80])]).astype(np.uint64)
    return flat, off


def _worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import conftest  # noqa: F401
    from kmer_extension_b200 import sharded
    from oracle import oracle as O
    try:
        sc = sharded.ShardedCounter(SpectrumStandIn(O), device=torch.device("cpu"))
        out = {}
        flat, off = _rows(rank)
        for k in (5, 21):
            hist, tail, info = sc.spectrum(torch.from_numpy(flat.copy()), int(off[-1]), torch.from_numpy(off.astype(np.int64)),
                                           len(off) - 1, k, hist_len=HIST_LEN)
            out[f"k{k}_hist"] = hist.numpy().view(np.uint64).copy()
            out[f"k{k}_tail"] = tail.numpy().view(np.uint64).copy()
        rows = ["ACGTACGTACGTACGTACGTAC", "ACGTNACGTACGTACGTACGTA" if rank == 1 else "ACGTTACGTACGTACGTACGTA"]
        fb, o2 = O.rows_to_flat(rows)
        raised = False
        try:
            sc.spectrum(torch.from_numpy(np.frombuffer(fb, np.uint8).copy()), int(o2[-1]), torch.from_numpy(o2.astype(np.int64)), 2, 15,
                        hist_len=HIST_LEN)
        except Exception:
            raised = True
        np.savez(Path(out_dir) / f"s{rank}.npz", raised=raised, **out)
    finally:
        dist.destroy_process_group()


def test_sharded_spectrum_two_ranks_gloo(tmp_path):
    import conftest  # noqa: F401
    import spectrum_util as S
    from oracle import oracle as O
    world = 2
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    outs = [np.load(tmp_path / f"s{r}.npz") for r in range(world)]
    assert all(bool(o["raised"]) for o in outs), "an input error on one rank must abort every rank"
    parts = [_rows(r) for r in range(world)]
    flat = np.concatenate([p[0] for p in parts])
    off = np.concatenate([parts[0][1], parts[1][1][1:] + parts[0][1][-1]])
    for k in (5, 21):
        keys, counts, n = O.np_count(flat, off, k)
        wh, wt = S.np_spectrum(keys, counts, HIST_LEN)
        assert wt.shape[0] > 0
        for o in outs:                                     # the same combined spectrum on every rank
            assert np.array_equal(o[f"k{k}_hist"], wh), k
            assert np.array_equal(S.sorted_tail(o[f"k{k}_tail"]), wt), k
