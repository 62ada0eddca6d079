"""GROUP BY kmer / count(*) on genome-sampled reads against the exact closed-form oracle (run on the B200 box: pytest -m gpu).

Reads drawn from one genome at some coverage, with substitution errors, are the input on which the counter changes paths:
  * low coverage (about 2x): many distinct repeated k-mers per bucket fill the leaf tables, and the k-mers that find a
    table full go to tier 2 as one-k-mer spill records;
  * higher coverage: buckets with more k-mers than fit on chip go to tier 2 as well, and tier 2 runs and fits;
  * higher still: tier 2 needs more than its table (tier2_decide_kernel), the device sets n_overflow and dev_finish
    recounts the whole batch through the global hash table (tier 3); the host entry points drop the groups that already
    streamed back;
  * sharded: every rank samples the same genome, so the high-count k-mers come from every source at once; an owner's
    tier 2 or a source's segment that does not fit raises KMER_ERR_CAPACITY, after which the owner merge counts exactly.
The oracle is tests/coverage_util.py (pinned by test_coverage_oracle.py), exact at 1 GB without sorting every window.

Every case asserts the regime it targets before it compares the table (n_tier2 / n_overflow from dev_finish, the
KMER_ERR_CAPACITY it expects, ShardedCounter's info["fallback"]).  The coverages were calibrated on one B200: if a later
change of the counter moves a regime's edge, resize the input, do not drop the precondition.
"""
import functools
import gc
import time

import numpy as np
import pytest

import coverage_util as CU
from kmer_extension_b200 import api
from oracle import oracle as O
from test_shard_regimes_gpu import _merge_fallback, count_owners, merge_owner, partition_sources, shard_owner

pytestmark = pytest.mark.gpu

MB = 1 << 20
READ_LEN = 1000


@pytest.fixture()
def eng():
    """A fresh context per test; prints the wall time and the peak device memory (torch's peak plus the workspaces the
    library allocates itself, noted by the test in eng.lib_bytes)."""
    import torch
    e = api.KmerCuda(0)
    e.lib_bytes = 0
    torch.cuda.reset_peak_memory_stats()
    t0 = time.time()
    yield e
    e.close()
    gc.collect()
    torch.cuda.empty_cache()
    peak = torch.cuda.max_memory_allocated()
    print(f"\n  {time.time() - t0:.1f} s, peak device memory {(peak + e.lib_bytes) / 2**30:.2f} GiB "
          f"(torch {peak / 2**30:.2f} + library workspaces {e.lib_bytes / 2**30:.2f})")


def _pow2_at_least(v):
    p = 1
    while p < v:
        p <<= 1
    return p


def note_workspaces(eng, n_kmers, k, recounted=False, ranks=1):
    """Bytes the library allocates for one count of n_kmers k-mers (records, spill list, failed-bucket ids and tier 2's
    table as count_part.cu sizes them; the tier-3 table when the batch was recounted)."""
    if k < 14:                                            # the dense path: one 8-byte bin per code
        eng.lib_bytes = max(eng.lib_bytes, 8 << (2 * k))
        return
    plan = eng.shard_plan(max(n_kmers, 1), k, ranks)
    recs = plan.n_buckets * plan.cap * plan.rec_bytes // ranks
    t2 = max(1 << 16, _pow2_at_least(n_kmers // 4)) * 16
    t3 = _pow2_at_least(max(1024, 2 * min(n_kmers, 4 ** k if k < 32 else n_kmers))) * 16 if recounted else 0
    eng.lib_bytes = max(eng.lib_bytes, recs + recs // 8 + plan.n_buckets * 12 + t2 + t3)


# ------------------------------------------------------------------ inputs and their oracle tables (cached: cases share them)

@functools.lru_cache(maxsize=1)
def reads(mb, cov, err, seed, read_len=READ_LEN):
    """About mb MiB of read_len-base reads at coverage cov of a genome of mb MiB / cov bases."""
    n_reads = (mb * MB) // read_len
    return CU.sample_reads(seed, int(n_reads * read_len / cov), n_reads, read_len, err)


@functools.lru_cache(maxsize=2)
def oracle(mb, cov, err, seed, k, read_len=READ_LEN):
    (flat, off), (genome, starts, err_pos) = reads(mb, cov, err, seed, read_len)
    return CU.coverage_table(genome, starts, np.diff(off.astype(np.int64)), err_pos, flat, k)


def upload(flat, off):
    import torch
    d_seq = torch.from_numpy(np.concatenate([flat, np.zeros(64, np.uint8)])).cuda()
    d_off = torch.from_numpy(np.asarray(off, np.int64).copy()).cuda()
    return d_seq, d_off


SIGN = -(1 << 63)


def device_sorted(d_keys, d_counts):
    """A device table (int64 tensors) -> numpy (keys, counts) in unsigned key order, sorted on the GPU."""
    import torch
    s, idx = torch.sort(d_keys ^ SIGN)
    return (s ^ SIGN).cpu().numpy().view(np.uint64), d_counts[idx].cpu().numpy().view(np.uint64)


def assert_exact(got_keys, got_counts, n_kmers, want, what):
    keys, counts, n = want
    assert n_kmers == n, (what, "k-mers counted != windows")
    assert got_keys.size == keys.size, (what, f"{got_keys.size} groups, want {keys.size}")
    assert np.array_equal(got_keys, keys), (what, "keys differ (a group split in two, or missing)")
    bad = np.flatnonzero(got_counts != counts)
    assert bad.size == 0, (what, f"{bad.size} counts differ, first {keys[bad[:3]]}: {got_counts[bad[:3]]} != {counts[bad[:3]]}")
    assert int(got_counts.sum(dtype=np.uint64)) == n


def regime_of(r):
    return "tier3" if r.n_overflow else ("tier2" if r.n_tier2 else "leaf")


# ------------------------------------------------------------------ 1. the single-GPU device API across coverage

# (mb, coverage, error rate, k, regime).  Calibrated on one B200; see the module docstring.
DEV = [
    # low coverage: leaf tables fill with distinct repeated k-mers (one-k-mer spill records to tier 2; 0.1-0.3 % of the k-mers)
    (64, 2, 0.002, 21, "tier2"), (64, 2, 0.002, 31, "tier2"), (64, 2, 0.002, 32, "tier2"),
    # tier 2 runs and fits (0.6 % of the k-mers at k = 14, 2-9 % at k >= 21)
    (128, 10, 0.002, 14, "tier2"), (128, 10, 0.002, 21, "tier2"), (128, 10, 0.002, 26, "tier2"), (128, 10, 0.002, 31, "tier2"),
    (128, 10, 0.002, 32, "tier2"),
    # tier 2 does not fit: the batch is recounted
    (128, 30, 0.002, 21, "tier3"), (128, 30, 0.002, 26, "tier3"), (128, 30, 0.002, 31, "tier3"), (128, 30, 0.002, 32, "tier3"),
    # 2 % errors: count-1 error k-mers and high-count genome k-mers in the same buckets (tier 2 fits up to k = 26)
    (128, 30, 0.02, 21, "tier2"), (128, 30, 0.02, 26, "tier2"), (128, 30, 0.02, 31, "tier3"),
    (256, 60, 0.002, 21, "tier3"),
    # k <= 13: the dense path's global table, the poly-T and poly-A bins far above the coverage
    (64, 30, 0.002, 13, "dense"),
]


@pytest.mark.parametrize("mb,cov,err,k,regime", DEV, ids=[f"{m}MB-cov{c}-err{e}-k{k}-{g}" for m, c, e, k, g in DEV])
def test_device_api_across_coverage(eng, mb, cov, err, k, regime):
    import torch
    (flat, off), _ = reads(mb, cov, err, 1)
    want = oracle(mb, cov, err, 1, k)
    n_rows, n_bases = len(off) - 1, int(off[-1])
    d_seq, d_off = upload(flat, off)
    cap = want[0].size + 4096
    pairs = torch.empty((cap, 2), dtype=torch.int64, device="cuda")
    uniq = torch.empty(cap, dtype=torch.int64, device="cuda")
    eng.dev_count(d_seq, n_bases, d_off, n_rows, k, pairs)
    r = eng.dev_finish()
    print(f"\n  {mb} MB, coverage {cov}x, errors {err}, k={k}: {r.n_kmers} k-mers, {r.n_distinct} groups, "
          f"n_tier2 {r.n_tier2} ({r.n_tier2 / r.n_kmers:.1%}), n_overflow {r.n_overflow}", end="")
    note_workspaces(eng, r.n_kmers, k, recounted=r.n_overflow > 0)
    if regime == "dense":
        assert r.n_tier2 == 0 and r.n_overflow == 0
        keys, counts = want[0], want[1]
        for run in (0, (1 << (2 * k)) - 1):      # poly-A, poly-T
            assert counts[np.searchsorted(keys, np.uint64(run))] > 10 * cov
    else:
        assert regime_of(r) == regime, f"the input was meant to reach {regime}: n_tier2 {r.n_tier2}, n_overflow {r.n_overflow}"
    assert_exact(*device_sorted(pairs[:r.n_distinct, 0], pairs[:r.n_distinct, 1]), r.n_kmers, want, "dev_count")
    if k < 14:
        return
    eng.dev_count_split(d_seq, n_bases, d_off, n_rows, k, uniq, pairs)
    r2 = eng.dev_finish()
    assert (regime_of(r2), r2.n_tier2, r2.n_overflow) == (regime, r.n_tier2, r.n_overflow), "split: another regime"
    keys = torch.cat([uniq[:r2.n_unique], pairs[:r2.n_distinct, 0]])
    counts = torch.cat([torch.ones(r2.n_unique, dtype=torch.int64, device="cuda"), pairs[:r2.n_distinct, 1]])
    assert_exact(*device_sorted(keys, counts), r2.n_kmers, want, "dev_count_split")


# ------------------------------------------------------------------ 2. the bench shape: 1e6 reads x 1000, k = 21

def test_bench_shape_1gb_exact(eng, corc):
    """1e6 reads of 1000 bases (the shape of tools/coverage_experiment.py) at 10x, where tier 2 fits.  At 30x these reads
    need the tier-3 recount (n_overflow 1, with or without substitutions), whose table would take 32 GiB at this size."""
    import torch
    k, n_reads, cov = 21, 1_000_000, 10
    t0 = time.time()
    (flat, off), (genome, starts, err_pos) = CU.sample_reads(11, n_reads * READ_LEN // cov, n_reads, READ_LEN, 0.002)
    want = CU.coverage_table(genome, starts, np.diff(off.astype(np.int64)), err_pos, flat, k)
    del genome, starts, err_pos
    t_oracle = time.time() - t0
    d_seq, d_off = upload(flat, off)
    pairs = torch.empty((want[0].size + 4096, 2), dtype=torch.int64, device="cuda")
    eng.dev_count(d_seq, int(off[-1]), d_off, len(off) - 1, k, pairs)
    r = eng.dev_finish()
    note_workspaces(eng, r.n_kmers, k, recounted=r.n_overflow > 0)
    print(f"\n  1e6 x 1000 at {cov}x, k={k}: {r.n_kmers} k-mers, {r.n_distinct} groups, n_tier2 {r.n_tier2} "
          f"({r.n_tier2 / r.n_kmers:.1%}), n_overflow {r.n_overflow}; input + oracle {t_oracle:.0f} s", end="")
    assert regime_of(r) == "tier2"
    keys, counts = device_sorted(pairs[:r.n_distinct, 0], pairs[:r.n_distinct, 1])
    assert_exact(keys, counts, r.n_kmers, want, "dev_count 1 GB")
    s, n = corc.multiset_checksum(flat, off, k)           # of the input rows, independent of coverage_table
    assert n == r.n_kmers and O.np_table_checksum(keys, counts) == s


# ------------------------------------------------------------------ 3. the host entry points (pipelined: 8 pieces, 8 bucket groups)

HOST = [(128, 10, "tier2"), (128, 30, "tier3")]


@pytest.mark.parametrize("mb,cov,regime", HOST, ids=[f"{m}MB-cov{c}-{g}" for m, c, g in HOST])
def test_host_entry_points(eng, mb, cov, regime):
    import torch
    k, err = 21, 0.002
    (flat, off), _ = reads(mb, cov, err, 2)
    want = oracle(mb, cov, err, 2, k)
    n_rows, n_bases = len(off) - 1, int(off[-1])
    plan = eng.shard_plan(n_bases, k, 1)
    assert n_bases >= 4 * MB and (plan.n_buckets << plan.fine_shift) >= 4096      # the pipelined branch, 8 groups
    # the regime, through the device API on the same rows (the host path counts them with the same plan)
    d_seq, d_off = upload(flat, off)
    pairs = torch.empty((want[0].size + 4096, 2), dtype=torch.int64, device="cuda")
    eng.dev_count(d_seq, n_bases, d_off, n_rows, k, pairs)
    r = eng.dev_finish()
    print(f"\n  {mb} MB, coverage {cov}x, k={k}: n_tier2 {r.n_tier2} ({r.n_tier2 / r.n_kmers:.1%}), n_overflow {r.n_overflow}",
          end="")
    assert regime_of(r) == regime
    del d_seq, d_off, pairs
    torch.cuda.empty_cache()
    note_workspaces(eng, r.n_kmers, k, recounted=r.n_overflow > 0)
    eng.lib_bytes += (n_bases + n_rows * 8) + r.n_kmers * 24          # the column, pairs and codes buffers of the call

    def check(parts, n, what):
        keys = np.concatenate([p[0] for p in parts])
        counts = np.concatenate([p[1] for p in parts])
        o = np.argsort(keys, kind="stable")
        assert_exact(keys[o], counts[o], n, want, what)

    keys, counts, n = eng.count_kmers(flat, k, off)
    check([(keys, counts)], n, "count_kmers")
    u, keys, counts, n = eng.count_kmers_split(flat, k, off)
    check([(u, np.ones(u.size, np.uint64)), (keys, counts)], n, "count_kmers_split")
    u, keys, counts, n, nb = eng.count_kmers_packed(flat, k, off)
    assert nb == (2 * k + 7) // 8
    check([(u, np.ones(u.size, np.uint64)), (keys, counts)], n, "count_kmers_packed")


# ------------------------------------------------------------------ 4. sharded, simulated on one GPU

def rank_split(flat, off, G):
    """G ranks, each with its own reads (a contiguous range of rows) of the same genome"""
    edges = np.linspace(0, len(off) - 1, G + 1).astype(np.int64)
    return [(flat[int(off[a]):int(off[b])], off[a:b + 1] - off[a]) for a, b in zip(edges[:-1], edges[1:])]


def check_owner_tables(tables, want, owner_of):
    """The owners' tables together == the oracle, no k-mer from two owners, every owner holds only its own k-mers."""
    keys = np.concatenate([t[0] for t in tables])
    counts = np.concatenate([t[1] for t in tables])
    o = np.argsort(keys, kind="stable")
    assert_exact(keys[o], counts[o], sum(t[2] for t in tables), want, "union of the owners")
    for owner, t in enumerate(tables):
        assert (owner_of(t[0]) == owner).all(), f"owner {owner} holds k-mers of another rank"


SHARD_MB, SHARD_LEN = 64, 300
# (ranks, k, coverage, regime)
SHARD = [(2, 21, 10, "tier2"), (4, 21, 10, "tier2"), (2, 31, 10, "tier2"), (4, 31, 10, "tier2"),
         (2, 21, 60, "capacity"), (4, 21, 60, "capacity"), (2, 31, 60, "capacity"), (4, 31, 60, "capacity")]


@pytest.mark.parametrize("G,k,cov,regime", SHARD, ids=[f"G{g}-k{k}-cov{c}-{r}" for g, k, c, r in SHARD])
def test_sharded_same_genome_on_every_rank(eng, G, k, cov, regime):
    err = 0.002
    (flat, off), _ = reads(SHARD_MB, cov, err, 3, SHARD_LEN)
    want = oracle(SHARD_MB, cov, err, 3, k, SHARD_LEN)
    ranks = rank_split(flat, off, G)
    plan = eng.shard_plan(want[2], k, G)
    note_workspaces(eng, want[2], k, ranks=G)
    if regime == "tier2":
        send = partition_sources(eng, plan, ranks)
        tables = count_owners(eng, plan, send, want[2], seed=G + k)
        del send
        t2 = [t[3] for t in tables]
        print(f"\n  {G} ranks, k={k}, coverage {cov}x: owners' n_tier2 {t2}", end="")
        assert sum(t2) > 0, "tier 2 was expected to run on the owners"
        check_owner_tables(tables, want, lambda c: shard_owner(c, plan))
        return
    import torch
    failed = []
    send = []
    for r, (f, o) in enumerate(ranks):
        d_seq, d_off = upload(f, o)
        recs = torch.empty(plan.recs_bytes_per_peer * G, dtype=torch.uint8, device="cuda")
        fill = torch.empty(plan.buckets_per_rank * G, dtype=torch.int64, device="cuda")
        eng.dev_shard_partition(d_seq, int(o[-1]), d_off, len(o) - 1, plan, recs, fill)
        try:
            eng.dev_finish()
        except api.KmerSqlError as e:
            assert e.status == api.KMER_ERR_CAPACITY, e
            failed.append(("segment", r))
        send.append((recs, fill))
    if not failed:
        rb, fb = plan.recs_bytes_per_peer, plan.buckets_per_rank
        pairs = torch.empty((want[2] // G + 65536, 2), dtype=torch.int64, device="cuda")
        for owner in range(G):
            eng.dev_shard_count(plan, torch.cat([s[0][owner * rb:(owner + 1) * rb] for s in send]),
                                torch.cat([s[1][owner * fb:(owner + 1) * fb] for s in send]), pairs)
            try:
                eng.dev_finish()
            except api.KmerSqlError as e:
                assert e.status == api.KMER_ERR_CAPACITY, e
                failed.append(("owner", owner))
        del pairs
    del send
    print(f"\n  {G} ranks, k={k}, coverage {cov}x: KMER_ERR_CAPACITY from {failed}", end="")
    assert failed, "a segment or an owner's tier 2 was expected to run out of room"
    tables = _merge_fallback(eng, ranks, k, seed=G * k)
    check_owner_tables(tables, want, lambda c: merge_owner(c, G))


@pytest.mark.parametrize("cov,fallback", [(10, False), (60, True)], ids=["tier2", "capacity"])
def test_sharded_counter_one_process(eng, cov, fallback):
    import torch
    from kmer_extension_b200.sharded import ShardedCounter
    k, err = 21, 0.002
    (flat, off), _ = reads(SHARD_MB, cov, err, 3, SHARD_LEN)
    want = oracle(SHARD_MB, cov, err, 3, k, SHARD_LEN)
    note_workspaces(eng, want[2], k)
    d_seq, d_off = upload(flat, off)
    pairs = torch.empty((want[0].size + 65536, 2), dtype=torch.int64, device="cuda")
    nd, nk, info = ShardedCounter(eng).count(d_seq, int(off[-1]), d_off, len(off) - 1, k, pairs)
    print(f"\n  ShardedCounter, k={k}, coverage {cov}x: fallback {info['fallback']}, tier2_kmers {info['tier2_kmers']}", end="")
    assert info["fallback"] == fallback
    if not fallback:
        assert info["tier2_kmers"] > 0
    assert_exact(*device_sorted(pairs[:nd, 0], pairs[:nd, 1]), nk, want, "ShardedCounter")
