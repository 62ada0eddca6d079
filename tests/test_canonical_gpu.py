"""Canonical k-mer counting on the GPU against the oracles of tests/canonical_util.py (run on the B200 box: pytest -m gpu).

A k-mer and its reverse complement are one group keyed by min(code, rc(code)).  Every case is compared exactly: tables with
the numpy canonical count, the folded closed-form coverage oracle, or -- at the 1 GB bench shape -- the GPU's strand-specific
table folded on the device with torch.  Spectra are compared with the numpy spectrum of the same canonical table.  Cases that
target a regime (tier 2, the tier-3 recount) assert it first, as tests/test_coverage_gpu.py does.
"""
import numpy as np
import pytest

import canonical_util as CN
import spectrum_util as S
from kmer_extension_b200 import api, datagen
from oracle import oracle as O
from test_coverage_gpu import device_sorted, eng, reads, regime_of, upload  # noqa: F401  (eng: fixture)

pytestmark = pytest.mark.gpu

FORMATS = ("pairs", "split", "spectrum")
HIST_LEN = 16


def mixed_rows(seed, n_rows=300, max_len=300, k=21):
    """ragged mixed-case random rows, rows of exactly k bases, poly-A / poly-T runs, and reverse-complement copies of rows"""
    rng = np.random.default_rng(seed)
    rows = []
    for _ in range(n_rows):
        n = int(rng.integers(k, max_len + 1))
        rows.append("".join("acgtACGT"[j] for j in rng.integers(0, 8, n)))
    rows += ["A" * (k + 40), "t" * (k + 25), "AC" * (k + 5), "acgt" * (k + 3)]
    rows += [CN.rc_text(r) for r in rows[:40]] + ["G" * k, "c" * k] + rows[:20]
    rows.append(rows[0][:k])
    return O.rows_to_flat(rows)


def dev_table(eng, flat, off, k, fmt, algo=api.ALGO_AUTO):
    """one canonical count through the device API in format fmt -> (sorted keys, counts, n_kmers) or ((hist, tail), n_kmers)"""
    import torch
    f = np.frombuffer(flat, np.uint8) if isinstance(flat, (bytes, bytearray)) else np.asarray(flat, np.uint8)
    d_seq, d_off = upload(f, off)
    n_rows, n_bases = len(off) - 1, int(off[-1])
    cap = max(eng.max_kmers(n_bases, n_rows, k), 1) + 64
    if fmt == "spectrum":
        hist = torch.full((HIST_LEN,), 0x5A5A, dtype=torch.int64, device="cuda")
        tail = torch.full((cap // HIST_LEN + 1, 2), 0x5A5A, dtype=torch.int64, device="cuda")
        eng.dev_count_spectrum(d_seq, n_bases, d_off, n_rows, k, hist, tail, algo, canonical=True)
        r = eng.dev_finish()
        return (hist.cpu().numpy().view(np.uint64).copy(), S.sorted_tail(tail[:r.n_distinct].cpu().numpy())), r
    pairs = torch.full((cap, 2), -1, dtype=torch.int64, device="cuda")
    if fmt == "pairs":
        eng.dev_count(d_seq, n_bases, d_off, n_rows, k, pairs, algo, canonical=True)
        r = eng.dev_finish()
        return device_sorted(pairs[:r.n_distinct, 0], pairs[:r.n_distinct, 1]), r
    uniq = torch.full((cap,), -1, dtype=torch.int64, device="cuda")
    if algo == api.ALGO_AUTO:
        eng.dev_count_split(d_seq, n_bases, d_off, n_rows, k, uniq, pairs, canonical=True)
    else:
        eng._check(eng.lib.kmer_cuda_dev_count_canonical(eng.ctx, d_seq.data_ptr(), n_bases, d_off.data_ptr(), n_rows, k,
                                                         uniq.data_ptr(), cap, pairs.data_ptr(), cap, algo, eng._stream_ptr()))
    r = eng.dev_finish()
    keys = torch.cat([uniq[:r.n_unique], pairs[:r.n_distinct, 0]])
    counts = torch.cat([torch.ones(r.n_unique, dtype=torch.int64, device="cuda"), pairs[:r.n_distinct, 1]])
    return device_sorted(keys, counts), r


def check(got, r, want, fmt, what):
    keys, counts, n = want
    assert r.n_kmers == n, (what, "k-mers counted != windows")
    if fmt == "spectrum":
        wh, wt = S.np_spectrum(keys, counts, HIST_LEN)
        h, t = got
        assert np.array_equal(h, wh), (what, h[:8], wh[:8])
        assert np.array_equal(t, wt), (what, "tail")
        return
    gk, gc = got
    assert np.array_equal(gk, keys), (what, f"{gk.size} groups, want {keys.size}")
    assert np.array_equal(gc, counts), what


def algos_for(k):
    a = [api.ALGO_HASH]
    if k <= 15:
        a.append(api.ALGO_DENSE)
    if k >= 14:
        a += [api.ALGO_PARTITION, api.ALGO_TWO_PASS]
    return a


# ------------------------------------------------------------------ 1. every k, algorithm and format (device and host)

KS = [1, 2, 3, 4, 6, 7, 8, 12, 13, 14, 15, 16, 20, 21, 22, 25, 26, 27, 28, 30, 31, 32]


@pytest.mark.parametrize("k", KS)
def test_every_k_algo_and_format(eng, k):
    flat, off = mixed_rows(k, k=k)
    want = CN.np_canonical_count(flat, off, k)
    for algo in algos_for(k) + [api.ALGO_AUTO]:
        for fmt in FORMATS:
            got, r = dev_table(eng, flat, off, k, fmt, algo)
            check(got, r, want, fmt, f"k={k} algo={algo} {fmt}")
    keys, counts, n = eng.count_kmers(flat, k, off, canonical=True)
    o = np.argsort(keys)
    assert n == want[2] and np.array_equal(keys[o], want[0]) and np.array_equal(counts[o], want[1]), "host pairs"
    u, pk, pc, n = eng.count_kmers_split(flat, k, off, canonical=True)
    keys = np.concatenate([u, pk])
    o = np.argsort(keys)
    assert np.array_equal(keys[o], want[0]) and np.array_equal(np.concatenate([np.ones(u.size, np.uint64), pc])[o], want[1]), "host split"
    h, t = eng.count_spectrum(flat, k, off, hist_len=HIST_LEN, canonical=True)
    wh, wt = S.np_spectrum(want[0], want[1], HIST_LEN)
    assert np.array_equal(h, wh) and np.array_equal(S.sorted_tail(t), wt), "host spectrum"


def test_known_answers(eng):
    for rows, k, want in ((["ACGTACGT"], 4, {"acgt": 2, "cgta": 2, "gtac": 1}), (["ACGTT"], 3, {"aac": 1, "acg": 2})):
        keys, counts, n = eng.count_kmers(rows, k, canonical=True)
        assert CN.counter_of(keys, counts, k) == want
    h, t = eng.count_spectrum(["ACGTACGT"], 4, hist_len=HIST_LEN, canonical=True)
    assert list(zip(*api.spectrum_rows(h, t))) == [(1, 1), (2, 2)]


# ------------------------------------------------------------------ 2. forced windows and an even-spread plan

WINDOWS = [(k, w) for k in (14, 18, 21, 22, 24, 25, 26) for w in (4, 6, 8, 9) if k - w + 1 >= 2] + \
          [(k, w) for k in (27, 28, 29, 31, 32) for w in (8, 12, 16)]


@pytest.mark.parametrize("k,w", WINDOWS)
def test_forced_windows(eng, k, w):
    """every minimizer window and record width, including those where the m-mer is capped (the centred canonical m-mers)"""
    flat, off = mixed_rows(100 + k + w, n_rows=400, max_len=400, k=k)
    want = CN.np_canonical_count(flat, off, k)
    eng.lib.kmer_cuda_test_force_window(w)
    try:
        for fmt in FORMATS:
            got, r = dev_table(eng, flat, off, k, fmt, api.ALGO_PARTITION)
            check(got, r, want, fmt, f"k={k} w={w} {fmt}")
    finally:
        eng.lib.kmer_cuda_test_force_window(0)


def test_even_spread_plan(eng):
    """k = 14 with window 9 forced: 4^6 / 2 canonical m-mers are fewer than 30 per bucket at 2e5 k-mers, so the plan spreads
    the m-mers over the buckets by a second hash (plan.even)"""
    flat, off = datagen.synth_reads(5, 1000, 220)
    flat = CN.revcomp_rows(flat, off, np.arange(1000) % 3 == 0)
    flat = np.concatenate([flat, flat[:int(off[300])]])
    off = np.concatenate([off, off[1:301] + off[-1]])
    k = 14
    assert 4 ** (k - 9 + 1) / 2 < 30 * (int(off[-1]) // 1200)
    want = CN.np_canonical_count(flat, off, k)
    eng.lib.kmer_cuda_test_force_window(9)
    try:
        for fmt in FORMATS:
            got, r = dev_table(eng, flat, off, k, fmt, api.ALGO_PARTITION)
            check(got, r, want, fmt, f"even {fmt}")
    finally:
        eng.lib.kmer_cuda_test_force_window(0)


# ------------------------------------------------------------------ 3. k = 32 edges and the reference's errors

def test_k32_all_a_all_t_and_mixed(eng):
    for rows in (["A" * 40] * 3, ["T" * 40] * 3, ["A" * 40, "t" * 50, "ACGT" * 20, "a" * 32, "T" * 32]):
        flat, off = O.rows_to_flat(rows)
        want = CN.np_canonical_count(flat, off, 32)
        for algo in (api.ALGO_HASH, api.ALGO_PARTITION):
            for fmt in FORMATS:
                got, r = dev_table(eng, flat, off, 32, fmt, algo)
                check(got, r, want, fmt, f"k=32 {rows[0][:3]} algo={algo} {fmt}")
        assert want[0][0] == 0


@pytest.mark.parametrize("rows,k", [(["ACGT", "ACGN", "AC"], 3), (["ACGTACGT", "AC", "ACGX"], 3), (["ACGTAC", "ACGTAC"], 33),
                                    (["ACGTAC"], 0), (["acgtacgtacgtacgtac", "ACGT-CGTACGTACGTACGT"], 14), (["A" * 30, "A" * 13], 14)])
def test_errors_are_the_strand_specific_ones(eng, rows, k):
    with pytest.raises(api.KmerSqlError) as want:
        eng.count_kmers(rows, k)
    for call in (lambda: eng.count_kmers(rows, k, canonical=True), lambda: eng.count_kmers_split(rows, k, canonical=True),
                 lambda: eng.count_spectrum(rows, k, hist_len=HIST_LEN, canonical=True)):
        with pytest.raises(api.KmerSqlError) as got:
            call()
        assert (got.value.status, got.value.sqlstate, got.value.row) == (want.value.status, want.value.sqlstate, want.value.row)


# ------------------------------------------------------------------ 4. reads from both strands: tier 2, the tier-3 recount

COV = [(128, 10, 0.002, 21, "tier2"), (128, 10, 0.002, 31, "tier2"), (128, 30, 0.002, 21, "tier3"), (64, 30, 0.002, 13, "dense")]


@pytest.mark.parametrize("mb,cov,err,k,regime", COV, ids=[f"{m}MB-cov{c}-k{k}-{g}" for m, c, e, k, g in COV])
def test_both_strands_across_coverage(eng, mb, cov, err, k, regime):
    n_reads = (mb << 20) // 1000
    (flat, off), want = CN.both_strands(1, n_reads * 1000 // cov, n_reads, 1000, k, err)
    for fmt in FORMATS:
        got, r = dev_table(eng, flat, off, k, fmt)
        print(f"\n  {mb} MB {cov}x k={k} {fmt}: n_tier2 {r.n_tier2} ({r.n_tier2 / r.n_kmers:.1%}), n_overflow {r.n_overflow}", end="")
        if regime != "dense":
            assert regime_of(r) == regime, f"the input was meant to reach {regime}: n_tier2 {r.n_tier2}, n_overflow {r.n_overflow}"
        check(got, r, want, fmt, f"{mb} MB {cov}x k={k} {fmt}")
    if regime == "dense":
        return
    # the pipelined host path (>= 4 MiB, k >= 14) in all three formats
    keys, counts, n = eng.count_kmers(flat, k, off, canonical=True)
    o = np.argsort(keys)
    assert n == want[2] and np.array_equal(keys[o], want[0]) and np.array_equal(counts[o], want[1]), "host pairs"
    u, pk, pc, n = eng.count_kmers_split(flat, k, off, canonical=True)
    keys = np.concatenate([u, pk])
    o = np.argsort(keys)
    assert np.array_equal(keys[o], want[0]) and np.array_equal(np.concatenate([np.ones(u.size, np.uint64), pc])[o], want[1])
    h, t = eng.count_spectrum(flat, k, off, hist_len=HIST_LEN, canonical=True)
    wh, wt = S.np_spectrum(want[0], want[1], HIST_LEN)
    assert np.array_equal(h, wh) and np.array_equal(S.sorted_tail(t), wt), "host spectrum"


@pytest.mark.parametrize("k", [13, 14, 21, 27, 32])
def test_strand_invariance(eng, k):
    """reverse-complementing any subset of the rows changes no result"""
    flat, off = datagen.synth_reads(17, 3000, 600)
    flat = np.concatenate([flat, flat[:int(off[1500])]])             # repeats, so tables and tails are not trivial
    off = np.concatenate([off, off[1:1501] + off[-1]])
    base = {fmt: dev_table(eng, flat, off, k, fmt)[0] for fmt in FORMATS}
    for seed in (1, 2):
        which = np.random.default_rng(seed).integers(0, 2, len(off) - 1).astype(bool)
        flat2 = CN.revcomp_rows(flat, off, which)
        for fmt in FORMATS:
            got = dev_table(eng, flat2, off, k, fmt)[0]
            assert all(np.array_equal(a, b) for a, b in zip(got, base[fmt])), (k, seed, fmt)


# ------------------------------------------------------------------ 5. the 1 GB bench shape against the folded GPU table

def _fold_on_device(keys, counts, k):
    """strand-specific (int64) table -> canonical (sorted keys, summed counts), all on the device"""
    import torch
    x = ~keys
    r = torch.zeros_like(keys)
    for i in range(k):
        r |= ((x >> (2 * (k - 1 - i))) & 3) << (2 * i)
    c = torch.minimum(keys, r)
    s, idx = torch.sort(c)
    cs = counts[idx]
    u, inv, n = torch.unique_consecutive(s, return_inverse=True, return_counts=True)
    tot = torch.zeros(u.numel(), dtype=torch.int64, device=keys.device).index_add_(0, inv, cs)
    return u, tot


def test_bench_shape_1gb_k21(eng):
    """1e6 uniform reads x 1000 bases generated in HBM (the bench workload), k = 21: the canonical table equals the GPU's
    strand-specific table (oracle-pinned by the other suites) folded with torch; the canonical spectrum equals that table's"""
    import torch
    k, n_rows, L = 21, 1_000_000, 1000
    d_seq = torch.empty(n_rows * L + 80, dtype=torch.uint8, device="cuda")
    d_off = torch.empty(n_rows + 1, dtype=torch.int64, device="cuda")
    eng.dev_synth_reads(2, 0, n_rows, L, d_seq, d_off)
    n = n_rows * (L - k + 1)
    pairs = torch.empty((n, 2), dtype=torch.int64, device="cuda")
    eng.dev_count(d_seq, n_rows * L, d_off, n_rows, k, pairs)
    r = eng.dev_finish()
    fk, fc = _fold_on_device(pairs[:r.n_distinct, 0], pairs[:r.n_distinct, 1], k)
    eng.dev_count(d_seq, n_rows * L, d_off, n_rows, k, pairs, canonical=True)
    rc = eng.dev_finish()
    assert rc.n_kmers == n and rc.n_distinct == fk.numel()
    s, idx = torch.sort(pairs[:rc.n_distinct, 0])
    assert torch.equal(s, fk) and torch.equal(pairs[:rc.n_distinct, 1][idx], fc)
    del s, idx
    hist = torch.empty(65536, dtype=torch.int64, device="cuda")
    tail = torch.empty((1024, 2), dtype=torch.int64, device="cuda")
    folded = torch.stack([fk, fc], dim=1).contiguous()
    eng.dev_pairs_spectrum(folded, folded.shape[0], hist, tail)
    rw = eng.dev_finish()
    wh, wt = hist.clone(), S.sorted_tail(tail[:rw.n_distinct].cpu().numpy())
    eng.dev_count_spectrum(d_seq, n_rows * L, d_off, n_rows, k, hist, tail, canonical=True)
    rs = eng.dev_finish()
    assert torch.equal(hist, wh) and np.array_equal(S.sorted_tail(tail[:rs.n_distinct].cpu().numpy()), wt)
    print(f"\n  1 GB k=21: {r.n_distinct} strand-specific groups, {rc.n_distinct} canonical; n_tier2 {r.n_tier2} / {rc.n_tier2}", end="")
