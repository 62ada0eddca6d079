"""The sharded counter in the regimes that small inputs never reach (run on the B200 box: pytest -m gpu).

The partition counter takes different code paths depending on the size of the WHOLE job and on the number of sources:
  * even spread: above ~1.7e8 k-mers at k = 14 the m-mers are too coarse for the buckets and are spread by a second hash
    (bucket_position<W>(h, even) -> mix32), on the source side (partition_kernel) and on the owner side (refine kernels);
  * chunked plans: n_src = n_ranks * chunks_per_rank segments per coarse partition, up to KMER_MAX_SRC = 32;
  * the refine kernel: refine_staged_kernel only for 8-byte records at fine_shift 8, refine_kernel<W, 1|2> otherwise;
  * the exact fallback for skewed input: every rank counts its own rows, the tables are merged by owner hash;
  * partition -> count chained on one context, the partition's findings reported by the count's finish;
  * the dense k <= 13 path split over many ranks.
A shard plan's total is a parameter: an inflated total reaches a large-job regime while the real rows stay small.

Every rank is simulated on one GPU: each source partitions into its own send buffer, and each owner's receive side is built
by slicing those buffers (the all-to-all) or by pointing straight into them (the peer read).  Every test asserts the plan
fields of the regime it means to cover first, then compares exactly with the oracle: the union of the owners' tables is the
GROUP BY table, no k-mer comes from two owners, and the owners' k-mer counts add up to the number of windows.
"""
import gc

import numpy as np
import pytest

from kmer_extension_b200 import api, datagen
from oracle import oracle as O

pytestmark = pytest.mark.gpu

GARBAGE = 0xA5      # fills every send buffer before the partition: only the filled part of a segment may be read


@pytest.fixture()
def eng():
    """A fresh context per test, so that one case's workspaces do not stay allocated during the next."""
    import torch
    e = api.KmerCuda(0)
    torch.cuda.reset_peak_memory_stats()
    yield e
    e.close()
    gc.collect()
    torch.cuda.empty_cache()
    print(f"\n  peak torch allocation {torch.cuda.max_memory_allocated() / 2**30:.2f} GiB")


# ------------------------------------------------------------------ inputs

def rows_flat(rows):
    flat, off = O.rows_to_flat(rows)
    return np.frombuffer(flat, np.uint8), off


def join(parts):
    """(flat, off) pieces -> one (flat, off) holding their rows in order."""
    parts = list(parts)
    flat = np.concatenate([p[0] for p in parts] + [np.zeros(0, np.uint8)])
    offs, base = [np.zeros(1, np.uint64)], np.uint64(0)
    for _, o in parts:
        offs.append(np.asarray(o[1:], np.uint64) + base)
        base += np.uint64(o[-1])
    return flat, np.concatenate(offs)


def rows_of(flat, off, r0, r1):
    return flat[int(off[r0]):int(off[r1])], off[r0:r1 + 1] - off[r0]


def cut_rows(flat, off, C, rng):
    """C pieces on row boundaries: C - 1 of them hold the rows in order, one EMPTY piece sits at a random position."""
    n = len(off) - 1
    assert n >= C - 1
    edges = np.linspace(0, n, C, dtype=np.int64)
    pieces = [rows_of(flat, off, int(edges[i]), int(edges[i + 1])) for i in range(C - 1)]
    pieces.insert(int(rng.integers(C)), (np.zeros(0, np.uint8), np.zeros(1, np.uint64)))
    return pieces


def windows(off, k):
    lens = np.diff(np.asarray(off, np.int64))
    return int(np.maximum(lens - k + 1, 0).sum())


def upload(flat, off):
    import torch
    d_seq = torch.from_numpy(np.concatenate([flat, np.zeros(64, np.uint8)])).cuda()   # 64 bytes of tail the kernels may read
    d_off = torch.from_numpy(np.asarray(off, np.int64).copy()).cuda()
    return d_seq, d_off


def sorted_table(keys, counts):
    o = np.argsort(keys, kind="stable")
    return keys[o], counts[o]


def read_pairs(pairs, n):
    p = pairs[:n].cpu().numpy().view(np.uint64)
    return p[:, 0].copy(), p[:, 1].copy()


# ------------------------------------------------------------------ restatements of the owner functions

def _u32(x):
    return np.asarray(x, np.uint64) & np.uint64(0xFFFFFFFF)


def _umulhi(a, b):
    return (_u32(a) * _u32(b)) >> np.uint64(32)


def _mmer_hash(top, himask, m):
    """common.cuh mmer_hash (32-bit wrap-around arithmetic in uint64)."""
    t = _u32((top & himask) * np.uint64(0x9E3779B1))
    t ^= (t >> np.uint64(m)) & himask
    t = _u32(t * np.uint64(0x85EBCA6B))
    t ^= (t >> np.uint64(m + 1)) & himask
    return t


def _mix32(x):
    x = _u32(x)
    x ^= x >> np.uint64(16)
    x = _u32(x * np.uint64(0x7FEB352D))
    x ^= x >> np.uint64(15)
    x = _u32(x * np.uint64(0x846CA68B))
    x ^= x >> np.uint64(16)
    return x


def _tent_position(h, W):
    """common.cuh bucket_position<W>(h): position of equal expected load, folded by the tent map."""
    v = _u32(~h)
    v2 = _umulhi(v, v)
    v4 = _umulhi(v2, v2)
    v8 = _umulhi(v4, v4)
    p = {4: v4, 6: _umulhi(v4, v2), 8: v8, 9: _umulhi(v8, v), 12: _umulhi(v8, v4), 16: _umulhi(v8, v8)}[W]
    F = _u32(~p)
    F = np.where(F >> np.uint64(31), _u32(~F), F)
    return _u32(F << np.uint64(1))


def shard_owner(codes, plan):
    """Rank that owns each k-mer under `plan`: the coarse partition of its minimizer's bucket position (the minimizer is the
    smallest mmer_hash over the k-mer's first w m-mers), divided by buckets_per_rank."""
    codes = np.asarray(codes, np.uint64)
    k, w, m = plan.k, plan.w, plan.m
    himask = np.uint64((0xFFFFFFFF << (32 - 2 * m)) & 0xFFFFFFFF)
    hmin = np.full(codes.shape, 0xFFFFFFFF, np.uint64)
    for j in range(w):
        mm = (codes >> np.uint64(2 * (k - j - m))) & np.uint64((1 << (2 * m)) - 1)
        hmin = np.minimum(hmin, _mmer_hash(_u32(mm << np.uint64(32 - 2 * m)), himask, m))
    pos = _mix32(hmin) if plan.even_spread else _tent_position(hmin, w)
    coarse = _umulhi(_u32(pos << np.uint64(plan.fine_shift)), plan.n_buckets)
    return (coarse // np.uint64(plan.buckets_per_rank)).astype(np.int64)


def merge_owner(codes, n_ranks):
    """Owner of a group in the merge by owner (count_hash.cu merge_pairs_kernel)."""
    h = O.np_mix64(np.asarray(codes, np.uint64) ^ np.uint64(0x9E3779B97F4A7C15)) >> np.uint64(32)
    return (h % np.uint64(n_ranks)).astype(np.int64)


def refine_kernel_of(plan):
    """The owner-side split kernel launch_refine picks for the plan."""
    if plan.recw == 1 and plan.fine_shift == 8:
        return "refine_staged"
    return f"refine<{plan.w},{plan.recw}>"


# ------------------------------------------------------------------ the simulated ranks

def partition_sources(eng, plan, sources):
    """Every source (rank * chunks_per_rank + chunk) partitions its rows into its own send buffer."""
    import torch
    G = plan.n_ranks
    send = []
    for flat, off in sources:
        d_seq, d_off = upload(flat, off)
        recs = torch.full((plan.recs_bytes_per_peer * G,), GARBAGE, dtype=torch.uint8, device="cuda")
        fill = torch.full((plan.buckets_per_rank * G,), 0x0F0F0F0F0F0F0F0F, dtype=torch.int64, device="cuda")
        eng.dev_shard_partition(d_seq, int(off[-1]), d_off, len(off) - 1, plan, recs, fill)
        r = eng.dev_finish()
        assert r.n_kmers == windows(off, plan.k)
        send.append((recs, fill))
    return send


def count_owners(eng, plan, send, n_windows, seed):
    """Every owner counts its buckets three ways: the exchanged layout (dev_shard_count, dev_shard_count_split) and the
    sources read in place (dev_shard_count_peers; split format on odd owners).  The sources come in a shuffled order every
    time.  The three tables must agree; returns [(keys, counts, n_kmers, n_tier2)] per owner."""
    import torch
    G = plan.n_ranks
    n_src = G * plan.chunks_per_rank
    assert len(send) == n_src
    rb, fb = plan.recs_bytes_per_peer, plan.buckets_per_rank
    rng = np.random.default_rng(seed)
    cap = n_windows + 16
    out = []
    for owner in range(G):
        order = rng.permutation(n_src)
        rr = torch.cat([send[s][0][owner * rb:(owner + 1) * rb] for s in order])
        rf = torch.cat([send[s][1][owner * fb:(owner + 1) * fb] for s in order])
        pairs = torch.empty((cap, 2), dtype=torch.int64, device="cuda")
        uniq = torch.empty(cap, dtype=torch.int64, device="cuda")
        eng.dev_shard_count(plan, rr, rf, pairs)
        r = eng.dev_finish()
        keys, counts = sorted_table(*read_pairs(pairs, r.n_distinct))
        eng.dev_shard_count_split(plan, rr, rf, uniq, pairs)
        r2 = eng.dev_finish()
        u = uniq[:r2.n_unique].cpu().numpy().view(np.uint64)
        pk, pc = read_pairs(pairs, r2.n_distinct)
        k2, c2 = sorted_table(np.concatenate([u, pk]), np.concatenate([np.ones(u.size, np.uint64), pc]))
        assert r2.n_kmers == r.n_kmers and np.array_equal(k2, keys) and np.array_equal(c2, counts), (owner, "split")
        del rr, rf
        order = rng.permutation(n_src)
        use_uniq = owner % 2 == 1
        eng.dev_shard_count_peers(plan, [send[s][0].data_ptr() + owner * rb for s in order],
                                  [send[s][1].data_ptr() + owner * fb * 8 for s in order], uniq if use_uniq else None, pairs)
        r3 = eng.dev_finish()
        pk, pc = read_pairs(pairs, r3.n_distinct)
        u = uniq[:r3.n_unique].cpu().numpy().view(np.uint64) if use_uniq else np.zeros(0, np.uint64)
        k3, c3 = sorted_table(np.concatenate([u, pk]), np.concatenate([np.ones(u.size, np.uint64), pc]))
        assert r3.n_kmers == r.n_kmers and np.array_equal(k3, keys) and np.array_equal(c3, counts), (owner, "peers")
        out.append((keys, counts, int(r.n_kmers), int(r.n_tier2)))
    return out


def check_union(tables, flat, off, k, owner_of=None):
    """Union of the owners' tables == oracle, no k-mer from two owners, sum of n_kmers == windows; optionally every owner
    holds exactly the k-mers owner_of assigns it."""
    ok, oc, on = O.np_count(flat, off, k)
    keys = np.concatenate([t[0] for t in tables])
    counts = np.concatenate([t[1] for t in tables])
    assert np.unique(keys).size == keys.size, "two owners reported the same k-mer"
    assert sum(t[2] for t in tables) == on == windows(off, k)
    keys, counts = sorted_table(keys, counts)
    assert np.array_equal(keys, ok) and np.array_equal(counts, oc)
    if owner_of is not None:
        for owner, t in enumerate(tables):
            assert (owner_of(t[0]) == owner).all(), f"owner {owner} holds k-mers the plan gives to another rank"


def sharded_exact(eng, plan, ranks, seed=0):
    """ranks[r] = the pieces rank r partitions (chunks_per_rank of them): partition, count every owner, check the union."""
    sources = [p for pieces in ranks for p in pieces]
    flat, off = join(sources)
    send = partition_sources(eng, plan, sources)
    tables = count_owners(eng, plan, send, windows(off, plan.k), seed)
    del send
    check_union(tables, flat, off, plan.k, lambda c: shard_owner(c, plan))
    return tables


def random_rows(seed, n_rows, max_len=400, min_len=40):
    return datagen.synth_ragged(seed, n_rows, max_len, min_len=min_len, mixed_case=seed % 2 == 1)


# ------------------------------------------------------------------ 1. even spread, sharded (inflated plan totals)

@pytest.mark.parametrize("k,w,total,G", [(14, 4, 200_000_000, 1), (14, 4, 200_000_000, 2), (14, 4, 200_000_000, 3),
                                         (27, 16, 800_000_000, 2)])
def test_even_spread_sharded(eng, k, w, total, G):
    forced = k == 27
    try:
        if forced:
            eng.lib.kmer_cuda_test_force_window(w)
        plan = eng.shard_plan(total, k, G)
        assert (plan.even_spread, plan.w, plan.recw, plan.fine_shift, plan.chunks_per_rank) == (1, w, 1 if k <= 26 else 2, 8, 1)
        ranks = []
        for r in range(G):
            repeats = ["A" * 6000, "ACGTTGCA" * 800] + (["A" * 6000] * 3 if r == 0 else [])
            ranks.append([join([random_rows(700 + 10 * G + r, 900), rows_flat(repeats)])])
        assert sum(windows(p[0][1], k) for p in ranks) < total // 100     # the real rows are tiny: most buckets are empty
        tables = sharded_exact(eng, plan, ranks, seed=G)
        # four copies of the homopolymer put >= 1400 records in one fine bucket (room for 840 at k = 14, 308 at k = 27)
        assert sum(t[3] for t in tables) > 0, "the repeats were expected to take tier 2"
    finally:
        eng.lib.kmer_cuda_test_force_window(0)


# ------------------------------------------------------------------ 2. even spread, one GPU (a real 1.8e8-k-mer job)

def _bincount_codes_fixed(flat, n_rows, L, k):
    """Oracle of n_rows fixed-length rows (the first n_rows * L bases): histogram of all 4^k codes."""
    c2 = O._CODE_LUT[flat[:n_rows * L]].reshape(n_rows, L)
    acc = np.zeros((n_rows, L - k + 1), np.uint32)
    for j in range(k):
        acc <<= np.uint32(2)
        acc |= c2[:, j:L - k + 1 + j]
    return np.bincount(acc.ravel(), minlength=4 ** k)


def test_even_spread_single_gpu(eng):
    import torch
    k, n_rows, L = 14, 182_000, 1000
    reads, _ = datagen.synth_reads(2024, n_rows, L)
    rep, rep_off = rows_flat(["A" * 6000, "ACGTTGCA" * 800, "GATTACA" * 900, "T" * 3000])
    flat, off = join([(reads, np.arange(n_rows + 1, dtype=np.uint64) * np.uint64(L)), (rep, rep_off)])
    n_kmers = windows(off, k)
    plan = eng.shard_plan(n_kmers, k, 1)      # make_partition_plan for the same total
    assert (plan.even_spread, plan.w, plan.recw) == (1, 4, 1)
    ref = _bincount_codes_fixed(flat, n_rows, L, k)
    ref += np.bincount(O.np_generate(rep, rep_off, k).astype(np.int64), minlength=4 ** k)
    assert int(ref.sum()) == n_kmers
    n_distinct = int(np.count_nonzero(ref))

    def check(parts, n, what):
        keys = np.concatenate([p[0] for p in parts])
        got = np.zeros(4 ** k, np.int64)
        for ks, cs in parts:
            got += np.bincount(ks.astype(np.int64), weights=cs.astype(np.float64), minlength=4 ** k).astype(np.int64)
        assert n == n_kmers, what
        assert keys.size == n_distinct, (what, "a k-mer was reported twice or is missing")
        assert np.array_equal(got, ref), what

    d_seq, d_off = upload(flat, off)
    cap = eng.max_kmers(int(off[-1]), len(off) - 1, k)
    pairs = torch.empty((cap, 2), dtype=torch.int64, device="cuda")
    for algo in (api.ALGO_AUTO, api.ALGO_PARTITION):
        eng.dev_count(d_seq, int(off[-1]), d_off, len(off) - 1, k, pairs, algo=algo)
        r = eng.dev_finish()
        check([read_pairs(pairs, r.n_distinct)], int(r.n_kmers), ("dev_count", algo))
        assert r.n_overflow == 0
    uniq = torch.empty(cap, dtype=torch.int64, device="cuda")
    eng.dev_count_split(d_seq, int(off[-1]), d_off, len(off) - 1, k, uniq, pairs)
    r = eng.dev_finish()
    u = uniq[:r.n_unique].cpu().numpy().view(np.uint64)
    check([(u, np.ones(u.size, np.uint64)), read_pairs(pairs, r.n_distinct)], int(r.n_kmers), "dev_count_split")
    del pairs, uniq, d_seq, d_off
    torch.cuda.empty_cache()
    u, keys, counts, n = eng.count_kmers_split(flat, k, off)       # the pipelined host path: its plan comes from the whole batch
    check([(u, np.ones(u.size, np.uint64)), (keys, counts)], n, "count_kmers_split")


# ------------------------------------------------------------------ 3. chunked plans (n_src up to 32)

CHUNKED = [(1, 2, 14, 0), (1, 2, 27, 0), (2, 2, 21, 0), (2, 2, 32, 0), (3, 5, 26, 0), (4, 8, 27, 0),
           (16, 2, 14, 5_000_000), (16, 2, 32, 0), (1, 32, 21, 400_000), (1, 32, 27, 0)]


@pytest.mark.parametrize("G,C,k,total", CHUNKED, ids=[f"G{g}xC{c}-k{k}" for g, c, k, _ in CHUNKED])
def test_chunked_plans(eng, G, C, k, total):
    rng = np.random.default_rng(31 * G + C + k)
    ranks, real = [], 0
    for r in range(G):
        flat, off = random_rows(1000 + 40 * G + r, max(2 * C, 48), max_len=300)
        if r == G - 1:   # a little repetition: tens of records in one segment, far below a segment's room
            extra = rows_flat(["ACGTTGCA" * 40, "A" * 500])
            flat, off = join([(flat, off), extra])
        real += windows(off, k)
        ranks.append(cut_rows(flat, off, C, rng))
    plan = eng.shard_plan(max(total, real), k, G, C)
    assert (plan.chunks_per_rank, plan.n_ranks * plan.chunks_per_rank) == (C, G * C)
    assert plan.recw == (1 if k <= 26 else 2)
    if total:   # the total was raised so that the write-combining split runs with all 32 sources
        assert plan.fine_shift == 8 and refine_kernel_of(plan) == "refine_staged" and G * C == 32
    sharded_exact(eng, plan, ranks, seed=G * C + k)


@pytest.mark.parametrize("split", [False, True], ids=["pairs", "split"])
def test_sharded_counter_chunks_2_in_one_process(eng, split):
    """ShardedCounter(chunks=2) on a world of one: the rows are partitioned in two pieces, the owner reads both segments."""
    import torch
    from kmer_extension_b200.sharded import ShardedCounter
    k = 21
    flat, off = join([random_rows(4242, 2000, max_len=500), rows_flat(["GATTACA" * 300, "A" * 2000])])
    d_seq, d_off = upload(flat, off)
    n = windows(off, k)
    pairs = torch.empty((n + 16, 2), dtype=torch.int64, device="cuda")
    uniq = torch.empty(n + 16, dtype=torch.int64, device="cuda") if split else None
    sc = ShardedCounter(eng, chunks=2)
    nd, nk, info = sc.count(d_seq, int(off[-1]), d_off, len(off) - 1, k, pairs, d_uniq=uniq)
    plan = info["plan"]
    assert not info["fallback"] and plan.chunks_per_rank == 2 and plan.n_ranks == 1
    keys, counts = read_pairs(pairs, nd)
    if split:
        u = uniq[:info["n_unique"]].cpu().numpy().view(np.uint64)
        keys, counts = np.concatenate([u, keys]), np.concatenate([np.ones(u.size, np.uint64), counts])
    check_union([(keys, counts, nk)], flat, off, k)


# ------------------------------------------------------------------ 4. fine_shift regimes and the refine kernel they select

FINE = [(21, 16, 19_200, 0, "refine<9,1>"), (31, 16, 19_200, 0, "refine<16,2>"),
        (21, 2, 24_000, 3, "refine<9,1>"), (31, 2, 24_000, 3, "refine<16,2>"),
        (21, 2, 400_000, 7, "refine<9,1>"), (31, 2, 400_000, 7, "refine<16,2>"),
        (21, 2, 700_000, 8, "refine_staged"), (31, 2, 700_000, 8, "refine<16,2>")]


@pytest.mark.parametrize("k,G,total,fine_shift,kernel", FINE, ids=[f"k{f[0]}-G{f[1]}-shift{f[3]}" for f in FINE])
def test_fine_shift_regimes(eng, k, G, total, fine_shift, kernel):
    max_len = 60 if G == 16 else 400
    n_rows = max(4, int(0.5 * total / G / ((40 + max_len) / 2 - k + 1)))   # the real rows fill about half of the plan's total
    ranks = []
    for r in range(G):
        flat, off = random_rows(1300 + 17 * fine_shift + r, n_rows, max_len=max_len)
        if r == 0:
            flat, off = join([(flat, off), rows_flat(["ACGTTGCA" * 40, "T" * 300])])
        ranks.append([(flat, off)])
    real = sum(windows(p[0][1], k) for p in ranks)
    assert real <= total
    plan = eng.shard_plan(total, k, G)
    assert (plan.fine_shift, plan.even_spread, refine_kernel_of(plan)) == (fine_shift, 0, kernel)
    sharded_exact(eng, plan, ranks, seed=fine_shift)


# ------------------------------------------------------------------ 5. segment overflow, then the merge by owner

def _merge_fallback(eng, rank_rows, k, seed):
    """sharded.py's exact fallback on simulated ranks: every rank counts its own rows on one GPU, every owner merges the
    groups it owns out of every rank's table (shuffled, plus an empty table).  Returns [(keys, counts, n_kmers)]."""
    import torch
    G = len(rank_rows)
    rng = np.random.default_rng(seed)
    local = []
    for flat, off in rank_rows:
        cap = max(eng.max_kmers(int(off[-1]), len(off) - 1, k), 1)
        t = torch.empty((cap, 2), dtype=torch.int64, device="cuda")
        n = 0
        if len(off) > 1:
            d_seq, d_off = upload(flat, off)
            eng.dev_count(d_seq, int(off[-1]), d_off, len(off) - 1, k, t)
            n = int(eng.dev_finish().n_distinct)
        local.append((t, n))
    empty = torch.empty((1, 2), dtype=torch.int64, device="cuda")
    max_groups = int(sum(n for _, n in local) / G * 1.3) + 65536       # sized as sharded.py sizes it
    out = []
    for owner in range(G):
        eng.dev_merge_begin(max_groups)
        adds = [local[i] for i in rng.permutation(G)]
        adds.insert(int(rng.integers(G + 1)), (empty, 0))
        for t, n in adds:
            eng.dev_merge_add(t, n, owner, G)
        pairs = torch.empty((max_groups, 2), dtype=torch.int64, device="cuda")
        eng.dev_merge_emit(k, pairs)
        r = eng.dev_finish()
        keys, counts = read_pairs(pairs, r.n_distinct)
        out.append((keys, counts, int(r.n_kmers)))
    return out


@pytest.mark.parametrize("G", [2, 3, 5, 16])
def test_overflow_then_owner_merge(eng, G):
    k = 21
    rank_rows = []
    for r in range(G):
        parts = [random_rows(1500 + 7 * G + r, 300 if G < 16 else 60)]
        if r == 1:
            parts.append(rows_flat(["A" * 200_000, "ACGT" * 500]))
        rank_rows.append(join(parts))
    total = sum(windows(o, k) for _, o in rank_rows)
    plan = eng.shard_plan(total, k, G)
    # the homopolymer's records all fall into one segment of rank 1: more than the segment holds
    import torch
    send = []
    for r, (flat, off) in enumerate(rank_rows):
        d_seq, d_off = upload(flat, off)
        recs = torch.empty(plan.recs_bytes_per_peer * G, dtype=torch.uint8, device="cuda")
        fill = torch.empty(plan.buckets_per_rank * G, dtype=torch.int64, device="cuda")
        eng.dev_shard_partition(d_seq, int(off[-1]), d_off, len(off) - 1, plan, recs, fill)
        if r == 1:
            with pytest.raises(api.KmerSqlError) as ei:
                eng.dev_finish()
            assert ei.value.status == api.KMER_ERR_CAPACITY
        else:
            eng.dev_finish()
        send.append((recs, fill))
    del send
    tables = _merge_fallback(eng, rank_rows, k, seed=G)
    flat, off = join(rank_rows)
    check_union(tables, flat, off, k, lambda c: merge_owner(c, G))
    assert all(t[0].size > 0 for t in tables), "every owner holds some of the thousands of distinct k-mers"


@pytest.mark.parametrize("G,with_random", [(3, True), (16, False)])
def test_owner_merge_k32_all_ones_code(eng, G, with_random):
    """'T' * 32 is the all-ones code, the merge table's empty key: it is counted beside the table (special_count), after the
    owner filter, so it must come back exactly once, from its owner, with the full count."""
    k = 32
    rank_rows = []
    for r in range(G):
        rows = ["T" * 40] * (r + 1) + ["t" * 33]
        parts = [rows_flat(rows)]
        if with_random:
            parts.append(random_rows(1700 + r, 100))
        rank_rows.append(join(parts))
    tables = _merge_fallback(eng, rank_rows, k, seed=G + 32)
    flat, off = join(rank_rows)
    check_union(tables, flat, off, k, lambda c: merge_owner(c, G))
    ones = np.uint64(0xFFFFFFFFFFFFFFFF)
    want = sum(9 * (r + 1) + 2 for r in range(G))
    holders = [i for i, t in enumerate(tables) if (t[0] == ones).any()]
    assert holders == [int(merge_owner([ones], G)[0])]
    t = tables[holders[0]]
    assert int(t[1][t[0] == ones][0]) == want
    if not with_random:   # one distinct k-mer over 16 ranks: every other owner comes back empty
        assert [i for i, t in enumerate(tables) if t[0].size] == holders


# ------------------------------------------------------------------ 6. partition -> count chained on one context per rank

def _chained(rank_rows, k, seed):
    """One context per simulated rank; on each, the partition is followed directly by that rank's owner count (no finish in
    between): the count's finish reports the partition's findings.  Returns per rank (keys, counts, n_kmers) or the error."""
    import torch
    G = len(rank_rows)
    total = sum(windows(o, k) for _, o in rank_rows)
    ctxs = [api.KmerCuda(0) for _ in range(G)]
    try:
        plan = ctxs[0].shard_plan(max(total, 1), k, G)
        rb, fb = plan.recs_bytes_per_peer, plan.buckets_per_rank
        send, keep = [], []
        for c, (flat, off) in zip(ctxs, rank_rows):
            d_seq, d_off = upload(flat, off)
            recs = torch.full((rb * G,), GARBAGE, dtype=torch.uint8, device="cuda")
            fill = torch.empty(fb * G, dtype=torch.int64, device="cuda")
            c.dev_shard_partition(d_seq, int(off[-1]), d_off, len(off) - 1, plan, recs, fill)
            send.append((recs, fill)); keep.append((d_seq, d_off))
        torch.cuda.synchronize()
        rng = np.random.default_rng(seed)
        cap = total + 16
        outs = []
        for owner, c in enumerate(ctxs):
            pairs = torch.empty((cap, 2), dtype=torch.int64, device="cuda")
            uniq = torch.empty(cap, dtype=torch.int64, device="cuda")
            order = rng.permutation(G)
            how = owner % 3
            if how == 0:
                c.dev_shard_count(plan, torch.cat([send[s][0][owner * rb:(owner + 1) * rb] for s in order]),
                                  torch.cat([send[s][1][owner * fb:(owner + 1) * fb] for s in order]), pairs)
            elif how == 1:
                c.dev_shard_count_split(plan, torch.cat([send[s][0][owner * rb:(owner + 1) * rb] for s in order]),
                                        torch.cat([send[s][1][owner * fb:(owner + 1) * fb] for s in order]), uniq, pairs)
            else:
                c.dev_shard_count_peers(plan, [send[s][0].data_ptr() + owner * rb for s in order],
                                        [send[s][1].data_ptr() + owner * fb * 8 for s in order], None, pairs)
            try:
                r = c.dev_finish()
            except api.KmerSqlError as e:
                outs.append(e)
                continue
            keys, counts = read_pairs(pairs, r.n_distinct)
            if how == 1:
                u = uniq[:r.n_unique].cpu().numpy().view(np.uint64)
                keys, counts = np.concatenate([u, keys]), np.concatenate([np.ones(u.size, np.uint64), counts])
            outs.append((keys, counts, int(r.n_kmers)))
        torch.cuda.synchronize()
        return plan, outs
    finally:
        for c in ctxs:
            c.close()


def _chained_ranks(G, k, seed):
    return [random_rows(seed + r, 120) for r in range(G)]


@pytest.mark.parametrize("G,k", [(3, 21), (4, 31)])
def test_chained_partition_then_count(G, k):
    rank_rows = _chained_ranks(G, k, 1900 + G)
    plan, outs = _chained(rank_rows, k, seed=G)
    flat, off = join(rank_rows)
    check_union(outs, flat, off, k, lambda c: shard_owner(c, plan))


def _replace_row(rank_rows, r, i, row):
    flat, off = rank_rows[r]
    before, after = rows_of(flat, off, 0, i), rows_of(flat, off, i + 1, len(off) - 1)
    rank_rows[r] = join([before, rows_flat([row]), after])


@pytest.mark.parametrize("fault", ["invalid_dna", "short_row", "segment_overflow"])
def test_chained_partition_errors_reach_the_count(fault):
    G, k = 3, 21
    rank_rows = _chained_ranks(G, k, 2100)
    if fault == "invalid_dna":
        _replace_row(rank_rows, 1, 7, "ACGT" * 10 + "N" + "ACGT" * 10)
        _replace_row(rank_rows, 1, 9, "ACG")             # a later short row: the bad byte's row comes first
        want = (api.KMER_ERR_INVALID_DNA, 7)
    elif fault == "short_row":
        _replace_row(rank_rows, 1, 11, "ACGT" * 5)       # 20 bases < k
        want = (api.KMER_ERR_INVALID_K, 11)
    else:
        _replace_row(rank_rows, 1, 3, "A" * 200_000)
        want = (api.KMER_ERR_CAPACITY, None)
    _, outs = _chained(rank_rows, k, seed=3)
    for r in (0, 2):
        if fault == "segment_overflow":   # the homopolymer's owner may run out of room too (sharded.py then falls back everywhere)
            assert not isinstance(outs[r], Exception) or outs[r].status == api.KMER_ERR_CAPACITY, (r, outs[r])
        else:                             # input errors are reported only by the context that partitioned the rows
            assert not isinstance(outs[r], Exception), (r, outs[r])
    e = outs[1]
    assert isinstance(e, api.KmerSqlError), fault
    assert e.status == want[0], (fault, e)
    if want[1] is not None:
        assert e.row == want[1], (fault, e.row)


# ------------------------------------------------------------------ 7. dense emit over many ranks

@pytest.mark.parametrize("G,k", [(3, 1), (16, 1), (3, 13), (16, 13)])
def test_dense_emit_many_ranks(eng, G, k):
    import torch
    shards = [random_rows(2300 + r, 60, max_len=300, min_len=16) for r in range(G)]
    table = torch.zeros(4 ** k, dtype=torch.int64, device="cuda")
    for flat, off in shards:
        d_seq, d_off = upload(flat, off)
        t = torch.empty(4 ** k, dtype=torch.int64, device="cuda")
        eng.dev_dense_table(d_seq, int(off[-1]), d_off, len(off) - 1, k, t)
        eng.dev_finish()
        table += t          # stands in for the all-reduce
        del t
    flat, off = join(shards)
    n_windows = windows(off, k)
    pairs = torch.empty((min(4 ** k, n_windows) + 16, 2), dtype=torch.int64, device="cuda")
    tables = []
    for rank in range(G):
        eng.dev_dense_emit(table, k, rank, G, pairs)
        r = eng.dev_finish()
        keys, counts = read_pairs(pairs, r.n_distinct)
        assert (keys % np.uint64(G) == np.uint64(rank)).all()
        tables.append((keys, counts, int(r.n_kmers)))
    check_union(tables, flat, off, k, lambda c: (c % np.uint64(G)).astype(np.int64))
    if k == 1:   # four bins: rank b % G emits bin b, ranks 4.. get nothing
        assert [t[0].size for t in tables] == [sum(1 for b in range(4) if b % G == r) for r in range(G)]
