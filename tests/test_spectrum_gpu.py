"""The k-mer abundance spectrum (count of counts) on the GPU against the oracles (run on the B200 box: pytest -m gpu).

kmer_cuda_dev_count_spectrum bins every group where it is counted -- the leaf's unique k-mers and table entries, tier 2 and
the tier-3 recount, the dense and hash paths, the k = 32 all-ones key -- instead of writing it.  Every case compares
  * hist and the tail (sorted) with the numpy spectrum of the GROUP BY (tests/spectrum_util.py) or of the closed-form coverage
    oracle, and/or with kmer_cuda_dev_pairs_spectrum of kmer_cuda_dev_count's table of the same rows;
  * the invariant sum(c * hist[c]) + sum(tail counts) = windows.
Output buffers are pre-filled with garbage: the library must overwrite the whole histogram.  Every regime case asserts the
regime it targets first (n_tier2, n_overflow, plan fields, KMER_ERR_CAPACITY), as test_coverage_gpu.py does.
"""
import numpy as np
import pytest

import coverage_util as CU
import spectrum_util as S
from kmer_extension_b200 import api, datagen
from oracle import oracle as O
from test_coverage_gpu import eng, note_workspaces, oracle, reads, regime_of, upload  # noqa: F401  (eng: fixture)
from test_shard_regimes_gpu import _merge_fallback, partition_sources

pytestmark = pytest.mark.gpu

GARBAGE = 0x5A5A5A5A5A5A5A5A


def windows(off, k):
    lens = np.diff(np.asarray(off, np.int64))
    return int(np.maximum(lens - (k - 1), 0).sum())


def out_buffers(hist_len, tail_cap):
    import torch
    return (torch.full((hist_len,), GARBAGE, dtype=torch.int64, device="cuda"),
            torch.full((tail_cap, 2), GARBAGE, dtype=torch.int64, device="cuda"))


def read_spectrum(hist, tail, r):
    return hist.cpu().numpy().view(np.uint64).copy(), S.sorted_tail(tail[:r.n_distinct].cpu().numpy())


def assert_spectrum(got, want, n_windows, what):
    (h, t), (wh, wt) = got, want
    assert h.size == wh.size and h[0] == 0, what
    bad = np.flatnonzero(h != wh)
    assert bad.size == 0, (what, f"bins {bad[:5]}: {h[bad[:5]]} != {wh[bad[:5]]}")
    assert np.array_equal(t, wt), (what, f"tail {t.shape[0]} groups, want {wt.shape[0]}")
    total = int((np.arange(h.size, dtype=np.uint64) * h).sum()) + int(t[:, 1].sum())
    assert total == n_windows, (what, "sum c * hist[c] + tail != windows")


def dev_spectrum(eng, d_seq, n_bases, d_off, n_rows, k, hist_len, tail_cap, algo=api.ALGO_AUTO):
    hist, tail = out_buffers(hist_len, tail_cap)
    eng.dev_count_spectrum(d_seq, n_bases, d_off, n_rows, k, hist, tail, algo)
    r = eng.dev_finish()
    assert r.n_unique == 0
    return read_spectrum(hist, tail, r), r


def pairs_spectrum_of_count(eng, d_seq, n_bases, d_off, n_rows, k, hist_len, algo=api.ALGO_AUTO):
    """dev_pairs_spectrum of dev_count's table of the same rows (the GPU-side cross-check)"""
    import torch
    pairs = torch.empty((max(eng.max_kmers(n_bases, n_rows, k), 1), 2), dtype=torch.int64, device="cuda")
    eng.dev_count(d_seq, n_bases, d_off, n_rows, k, pairs, algo)
    r = eng.dev_finish()
    hist, tail = out_buffers(hist_len, max(int(r.n_kmers) // hist_len, 1))
    eng.dev_pairs_spectrum(pairs, r.n_distinct, hist, tail)
    r2 = eng.dev_finish()
    assert r2.n_kmers == r.n_kmers
    return read_spectrum(hist, tail, r2), r


def np_want(flat, off, k, hist_len):
    keys, counts, n = O.np_count(flat, off, k)
    return S.np_spectrum(keys, counts, hist_len), n


def mixed_rows(seed, k):
    """ragged random reads, mixed case, plus repetition: poly-A and poly-T runs, one read forty times"""
    flat, off = datagen.synth_ragged(seed, 400, 300, min_len=max(k, 20), mixed_case=True)
    rep = flat[int(off[3]):int(off[4])]
    extra = [np.frombuffer(b"A" * 300, np.uint8), np.frombuffer(b"t" * 257, np.uint8)] + [rep] * 40
    parts = [flat] + extra
    offs = list(off) + list(int(off[-1]) + np.cumsum([e.size for e in extra]))
    return np.concatenate(parts), np.asarray(offs, np.uint64)


# ------------------------------------------------------------------ 1. every k, every algorithm, random and repetitive rows

@pytest.mark.parametrize("k", list(range(1, 33)))
def test_every_k_every_algo(eng, k):
    flat, off = mixed_rows(40 + k, k)
    d_seq, d_off = upload(flat, off)
    n_bases, n_rows = int(off[-1]), len(off) - 1
    hist_len = 64
    want, n = np_want(flat, off, k, hist_len)
    assert want[1].shape[0] > 0                                       # the repeats reach the tail
    tail_cap = n // hist_len
    algos = [api.ALGO_AUTO, api.ALGO_HASH] + ([api.ALGO_PARTITION, api.ALGO_TWO_PASS] if k >= 14 else [])
    for algo in algos:
        got, r = dev_spectrum(eng, d_seq, n_bases, d_off, n_rows, k, hist_len, tail_cap, algo)
        assert r.n_kmers == n and r.n_distinct == want[1].shape[0]
        assert_spectrum(got, want, n, f"k={k} algo={algo}")
        cross, _ = pairs_spectrum_of_count(eng, d_seq, n_bases, d_off, n_rows, k, hist_len, algo)
        assert_spectrum(cross, want, n, f"k={k} algo={algo} dev_pairs_spectrum(dev_count)")


@pytest.mark.parametrize("k,w", [(21, 4), (21, 6), (21, 8), (21, 9), (31, 8), (31, 12), (31, 16)])
def test_forced_minimizer_windows(eng, k, w):
    flat, off = mixed_rows(70 + w, k)
    d_seq, d_off = upload(flat, off)
    want, n = np_want(flat, off, k, 16)
    eng.lib.kmer_cuda_test_force_window(w)
    try:
        got, r = dev_spectrum(eng, d_seq, int(off[-1]), d_off, len(off) - 1, k, 16, n // 16, api.ALGO_PARTITION)
    finally:
        eng.lib.kmer_cuda_test_force_window(0)
    assert_spectrum(got, want, n, f"k={k} w={w}")


# ------------------------------------------------------------------ 2. histogram length edges and the tail's capacity

@pytest.mark.parametrize("hist_len", [2, 3, 1920, 1921, 65536])
@pytest.mark.parametrize("k", [13, 21, 32])
def test_hist_len_edges_and_tail_capacity(eng, k, hist_len):
    """hist_len 2: every repeated k-mer goes to the tail; 1920/1921: the largest count of a leaf table entry; the tail holds
    exactly the oracle's groups with count >= hist_len.  A tail one entry short fails with KMER_ERR_CAPACITY."""
    flat, off = mixed_rows(500 + k, k)
    # one k-mer 1920 times and one 1921 times (the leaf's largest table count and one more): homopolymer rows
    flat = np.concatenate([flat, np.frombuffer(b"C" * (1919 + k), np.uint8), np.frombuffer(b"G" * (1920 + k), np.uint8)])
    off = np.concatenate([off, [off[-1] + 1919 + k, off[-1] + 1919 + k + 1920 + k]]).astype(np.uint64)
    d_seq, d_off = upload(flat, off)
    n_bases, n_rows = int(off[-1]), len(off) - 1
    want, n = np_want(flat, off, k, hist_len)
    nt = want[1].shape[0]
    assert (nt > 0) == (hist_len <= 1921)
    got, r = dev_spectrum(eng, d_seq, n_bases, d_off, n_rows, k, hist_len, nt)
    assert r.n_distinct == nt
    assert_spectrum(got, want, n, f"k={k} hist_len={hist_len}, exact tail")
    assert nt <= n // hist_len                                        # what the header promises always suffices
    if not nt:
        return
    hist, tail = out_buffers(hist_len, nt - 1)
    eng.dev_count_spectrum(d_seq, n_bases, d_off, n_rows, k, hist, tail)
    with pytest.raises(api.KmerSqlError) as ei:
        eng.dev_finish()
    assert ei.value.status == api.KMER_ERR_CAPACITY and "output buffer too small" in ei.value.message


@pytest.mark.parametrize("t_count", [5, 63, 64, 65, 700])
def test_k32_all_ones_code(eng, t_count):
    """The k = 32 code of 't' * 32 is the hash tables' empty key, counted beside them: binned below hist_len, in the tail at
    or above it -- on the partition path and the hash path."""
    k, hist_len = 32, 64
    flat, off = datagen.synth_ragged(9, 200, 200, min_len=40, mixed_case=False)
    flat = np.concatenate([flat, np.frombuffer(b"T" * (t_count + 31), np.uint8)])
    off = np.concatenate([off, [off[-1] + t_count + 31]]).astype(np.uint64)
    d_seq, d_off = upload(flat, off)
    want, n = np_want(flat, off, k, hist_len)
    ones = np.uint64(0xFFFFFFFFFFFFFFFF)
    if t_count >= hist_len:
        assert ones in want[1][:, 0]
    for algo in (api.ALGO_PARTITION, api.ALGO_HASH):
        got, r = dev_spectrum(eng, d_seq, int(off[-1]), d_off, len(off) - 1, k, hist_len, n // hist_len + 1, algo)
        assert_spectrum(got, want, n, f"t*{t_count} algo={algo}")


# ------------------------------------------------------------------ 3. tiers: leaf tables full, tier 2, the tier-3 recount

# (mb, coverage, error rate, k, regime); calibrated in test_coverage_gpu.py.  At 2x many distinct repeated k-mers fill leaf
# tables (more than 1023 in a bucket: one-k-mer spill records to tier 2).
COV = [(64, 2, 0.002, 21, "tier2"), (128, 10, 0.002, 21, "tier2"), (128, 10, 0.002, 32, "tier2"), (128, 30, 0.002, 21, "tier3"),
       (128, 30, 0.002, 31, "tier3")]


@pytest.mark.parametrize("mb,cov,err,k,regime", COV, ids=[f"{m}MB-cov{c}-k{k}-{g}" for m, c, e, k, g in COV])
def test_tiers_against_the_coverage_oracle(eng, mb, cov, err, k, regime):
    (flat, off), _ = reads(mb, cov, err, 1)
    keys, counts, n = oracle(mb, cov, err, 1, k)
    d_seq, d_off = upload(flat, off)
    hist_len = 1024
    want = S.np_spectrum(keys, counts, hist_len)
    got, r = dev_spectrum(eng, d_seq, int(off[-1]), d_off, len(off) - 1, k, hist_len, n // hist_len)
    note_workspaces(eng, r.n_kmers, k, recounted=r.n_overflow > 0)
    print(f"\n  {mb} MB at {cov}x, k={k}: n_tier2 {r.n_tier2}, n_overflow {r.n_overflow}, tail {r.n_distinct}", end="")
    assert regime_of(r) == regime, f"the input was meant to reach {regime}"
    assert_spectrum(got, want, n, f"{mb} MB at {cov}x k={k}")


def test_bench_shape_1gb_at_10x(eng):
    """1e6 reads x 1000 bases at 10x coverage (tier 2 fits; at 30x the batch needs the 32 GiB tier-3 table)"""
    import torch
    k, n_reads, cov = 21, 1_000_000, 10
    (flat, off), _ = CU.sample_reads(11, n_reads * 1000 // cov, n_reads, 1000, 0.002)
    d_seq, d_off = upload(flat, off)
    n_bases, n_rows, n = int(off[-1]), len(off) - 1, windows(off, k)
    got, r = dev_spectrum(eng, d_seq, n_bases, d_off, n_rows, k, 65536, n // 65536)
    assert regime_of(r) == "tier2" and r.n_kmers == n
    cross, _ = pairs_spectrum_of_count(eng, d_seq, n_bases, d_off, n_rows, k, 65536)
    note_workspaces(eng, n, k)
    eng.lib_bytes += n * 16
    assert_spectrum(got, cross, n, "1 GB at 10x")
    del d_seq, d_off
    torch.cuda.empty_cache()


def test_uniform_bench_workload(eng):
    """the bench workload: 1e6 x 1000 uniform reads of seed 2, generated in HBM, k = 21"""
    import torch
    k, n_rows, L = 21, 1_000_000, 1000
    d_seq = torch.empty(n_rows * L + 80, dtype=torch.uint8, device="cuda")
    d_off = torch.empty(n_rows + 1, dtype=torch.int64, device="cuda")
    eng.dev_synth_reads(2, 0, n_rows, L, d_seq, d_off)
    n = n_rows * (L - k + 1)
    got, r = dev_spectrum(eng, d_seq, n_rows * L, d_off, n_rows, k, 65536, 1024)
    cross, _ = pairs_spectrum_of_count(eng, d_seq, n_rows * L, d_off, n_rows, k, 65536)
    note_workspaces(eng, n, k)
    eng.lib_bytes += n * 16
    assert r.n_kmers == n and got[0][1] > 0.99 * n
    assert_spectrum(got, cross, n, "uniform 1e6 x 1000")


# ------------------------------------------------------------------ 4. errors and empty input: exactly dev_count's

ERR_ROWS = [(["ACGTACGTACGTACGTACGTACGTA", "ACGTNACGTACGTACGTACGTACGT"], 21), (["ACGTACGTACGTACGTACGTACGTA", "ACGT"], 21),
            (["ACGTACGT", "ACGTAXGT", "AC"], 5), (["ACGTACGTACGTACGTACGTACGTACGTACGTACGT"], 33), (["ACGTACGTACGT"], 0),
            (["", "ACGTACGT"], 3)]


@pytest.mark.parametrize("rows,k", ERR_ROWS)
def test_errors_equal_dev_counts(eng, rows, k):
    import torch
    fb, off = O.rows_to_flat(rows)
    flat = np.frombuffer(fb, np.uint8)
    d_seq, d_off = upload(flat, off)
    pairs = torch.empty((64, 2), dtype=torch.int64, device="cuda")
    with pytest.raises(api.KmerSqlError) as want:
        eng.dev_count(d_seq, int(off[-1]), d_off, len(off) - 1, k, pairs)
        eng.dev_finish()
    hist, tail = out_buffers(8, 64)
    with pytest.raises(api.KmerSqlError) as got:
        eng.dev_count_spectrum(d_seq, int(off[-1]), d_off, len(off) - 1, k, hist, tail)
        eng.dev_finish()
    w, g = want.value, got.value
    assert (g.status, g.sqlstate, g.message, g.detail, g.row) == (w.status, w.sqlstate, w.message, w.detail, w.row)


def test_empty_input(eng):
    import torch
    d_seq = torch.zeros(64, dtype=torch.uint8, device="cuda")
    d_off = torch.zeros(1, dtype=torch.int64, device="cuda")
    hist, tail = out_buffers(16, 4)
    eng.dev_count_spectrum(d_seq, 0, d_off, 0, 21, hist, tail)
    r = eng.dev_finish()
    assert r.n_kmers == 0 and r.n_distinct == 0 and not hist.any()
    h, t = eng.count_spectrum([], 21, hist_len=16)
    assert h.size == 16 and not h.any() and t.shape == (0, 2)
    with pytest.raises(api.KmerSqlError) as ei:
        eng.count_spectrum([""], 21)
    assert ei.value.sqlstate == "22023" and ei.value.row == 0


# ------------------------------------------------------------------ 5. the host-buffer call, both regimes

@pytest.mark.parametrize("mb,cov,regime", [(2, 10, "small"), (128, 10, "tier2"), (128, 30, "tier3")])
def test_count_spectrum_host_path(eng, mb, cov, regime):
    k, err = 21, 0.002
    (flat, off), _ = reads(mb, cov, err, 1)
    keys, counts, n = oracle(mb, cov, err, 1, k)
    n_bases = int(off[-1])
    assert (n_bases >= 4 << 20) == (regime != "small")                 # the pipelined branch from 4 MiB on
    if regime != "small":
        d_seq, d_off = upload(flat, off)
        (_, r) = dev_spectrum(eng, d_seq, n_bases, d_off, len(off) - 1, k, 64, n // 64)
        assert regime_of(r) == regime
        del d_seq, d_off
    for hist_len in (64, 65536):
        h, t = eng.count_spectrum(flat, k, off, hist_len=hist_len)
        assert_spectrum((h, S.sorted_tail(t)), S.np_spectrum(keys, counts, hist_len), n, f"count_spectrum {mb} MB hist_len {hist_len}")
    c, m = api.spectrum_rows(h, t)
    wc, wm = np.unique(counts, return_counts=True)
    assert np.array_equal(c, wc) and np.array_equal(m, wm.astype(np.uint64))


# ------------------------------------------------------------------ 6. sharded, ranks simulated on one GPU

def _sum_owner_spectra(spectra, hist_len):
    hist = np.zeros(hist_len, np.uint64)
    for h, _ in spectra:
        hist += h
    tails = [t for _, t in spectra]
    return hist, S.sorted_tail(np.concatenate(tails) if tails else np.zeros((0, 2), np.uint64))


@pytest.mark.parametrize("G,k", [(2, 21), (4, 31)])
def test_sharded_owner_spectra(eng, G, k):
    """pull form (the sources' send buffers in place) and receive-buffer form (pointers into the exchanged layout): the owners'
    spectra sum to the oracle's, and agree form by form"""
    import torch
    err, cov, hist_len = 0.002, 10, 128
    (flat, off), _ = reads(64, cov, err, 3, 300)
    keys, counts, n = oracle(64, cov, err, 3, k, 300)
    edges = np.linspace(0, len(off) - 1, G + 1).astype(np.int64)
    ranks = [(flat[int(off[a]):int(off[b])], off[a:b + 1] - off[a]) for a, b in zip(edges[:-1], edges[1:])]
    plan = eng.shard_plan(n, k, G)
    assert plan.n_ranks == G and plan.chunks_per_rank == 1
    note_workspaces(eng, n, k, ranks=G)
    send = partition_sources(eng, plan, ranks)
    rb, fb = plan.recs_bytes_per_peer, plan.buckets_per_rank
    pull, recv, t2 = [], [], []
    for owner in range(G):
        hist, tail = out_buffers(hist_len, n // hist_len)
        eng.dev_shard_count_spectrum(plan, [s[0].data_ptr() + owner * rb for s in send],
                                     [s[1].data_ptr() + owner * fb * 8 for s in send], hist, tail)
        r = eng.dev_finish()
        t2.append(int(r.n_tier2))
        pull.append(read_spectrum(hist, tail, r))
        rr = torch.cat([s[0][owner * rb:(owner + 1) * rb] for s in send[::-1]])
        rf = torch.cat([s[1][owner * fb:(owner + 1) * fb] for s in send[::-1]])
        hist, tail = out_buffers(hist_len, n // hist_len)
        eng.dev_shard_count_spectrum(plan, [rr.data_ptr() + s * rb for s in range(G)], [rf.data_ptr() + s * fb * 8 for s in range(G)],
                                     hist, tail)
        r2 = eng.dev_finish()
        recv.append(read_spectrum(hist, tail, r2))
        assert np.array_equal(recv[-1][0], pull[-1][0]) and np.array_equal(recv[-1][1], pull[-1][1]), owner
    assert sum(t2) > 0, "tier 2 was expected to run on the owners"
    assert_spectrum(_sum_owner_spectra(pull, hist_len), S.np_spectrum(keys, counts, hist_len), n, f"{G} owners")


def test_sharded_capacity_fallback_spectra(eng):
    """60x coverage: the owners run out of room; the owner merge, emitted, then dev_pairs_spectrum per owner"""
    import torch
    G, k, hist_len = 3, 21, 256
    (flat, off), _ = reads(64, 60, 0.002, 3, 300)
    keys, counts, n = oracle(64, 60, 0.002, 3, k, 300)
    edges = np.linspace(0, len(off) - 1, G + 1).astype(np.int64)
    ranks = [(flat[int(off[a]):int(off[b])], off[a:b + 1] - off[a]) for a, b in zip(edges[:-1], edges[1:])]
    tables = _merge_fallback(eng, ranks, k, seed=5)
    spectra = []
    for tk, tc, _ in tables:
        pairs = torch.from_numpy(np.stack([tk, tc], axis=1).view(np.int64).copy()).cuda()
        hist, tail = out_buffers(hist_len, n // hist_len)
        eng.dev_pairs_spectrum(pairs, tk.size, hist, tail)
        spectra.append(read_spectrum(hist, tail, eng.dev_finish()))
    assert_spectrum(_sum_owner_spectra(spectra, hist_len), S.np_spectrum(keys, counts, hist_len), n, "merge fallback")


@pytest.mark.parametrize("k", [1, 9, 13])
def test_sharded_dense_spectra(eng, k):
    import torch
    G, hist_len = 3, 32
    parts = [mixed_rows(300 + r, k) for r in range(G)]
    flat = np.concatenate([p[0] for p in parts])
    offs = [np.zeros(1, np.uint64)]
    for p in parts:
        offs.append(p[1][1:] + offs[-1][-1])
    off = np.concatenate(offs)
    want, n = np_want(flat, off, k, hist_len)
    table = torch.zeros(1 << (2 * k), dtype=torch.int64, device="cuda")
    for f, o in parts:
        t = torch.empty_like(table)
        d_seq, d_off = upload(f, o)
        eng.dev_dense_table(d_seq, int(o[-1]), d_off, len(o) - 1, k, t)
        eng.dev_finish()
        table += t
    spectra = []
    for rank in range(G):
        pairs = torch.empty(((1 << (2 * k)) // G + 1, 2), dtype=torch.int64, device="cuda")
        eng.dev_dense_emit(table, k, rank, G, pairs)
        nd = eng.dev_finish().n_distinct
        hist, tail = out_buffers(hist_len, n // hist_len)
        eng.dev_pairs_spectrum(pairs, nd, hist, tail)
        spectra.append(read_spectrum(hist, tail, eng.dev_finish()))
    assert_spectrum(_sum_owner_spectra(spectra, hist_len), want, n, f"dense k={k}")


@pytest.mark.parametrize("k,cov,fallback", [(21, 10, False), (21, 60, True), (11, 10, False)])
def test_sharded_counter_spectrum_one_process(eng, k, cov, fallback):
    from kmer_extension_b200.sharded import ShardedCounter
    (flat, off), _ = reads(64, cov, 0.002, 3, 300)
    keys, counts, n = oracle(64, cov, 0.002, 3, k, 300)
    note_workspaces(eng, n, k)
    d_seq, d_off = upload(flat, off)
    hist, tail, info = ShardedCounter(eng).spectrum(d_seq, int(off[-1]), d_off, len(off) - 1, k, hist_len=512)
    assert info["fallback"] == fallback
    got = (hist.cpu().numpy().view(np.uint64).copy(), S.sorted_tail(tail.cpu().numpy()))
    assert_spectrum(got, S.np_spectrum(keys, counts, 512), n, f"ShardedCounter.spectrum k={k} at {cov}x")
