"""The host-buffer GROUP BY at the sizes real columns have, and the output-capacity contract of the device API.

kmer_cuda_submit_count / _split / _packed take one of two branches (submit_count_common, api.cu):
  * plain: upload, count, finish, download -- k <= 13 or fewer than 4 MiB bases;
  * pipelined: 14 <= k <= 32 and at least 4 MiB bases.  The column goes up in 8 pieces cut on tile boundaries (each copied
    with the 64 bytes behind it and partitioned on its own), the buckets are counted in 1 or 8 groups, and the finished part
    of the result streams back behind every group while later groups still count.  Tier 2's groups and the k == 32 key
    't'*32 leave after the last group; a tier-3 recount replaces what already left.
Every result here is compared bit for bit with the numpy oracle, and the launch count of each call pins the branch it took.

The device entry points take the capacity of their output (numel() of the tensor view handed in); a result that does not
fit must raise KMER_ERR_CAPACITY without writing past the view.
"""
import numpy as np
import pytest

from kmer_extension_b200 import api, datagen
from oracle import oracle as O

pytestmark = pytest.mark.gpu

MiB = 1 << 20
TILE = 4096                   # bases per tile (scan.cuh)
PIPELINE_MIN_BASES = 4 * MiB  # smallest column the pipelined branch takes
KS = (14, 21, 22, 26, 27, 31, 32)
SPECIAL = np.uint64(0xFFFFFFFFFFFFFFFF)   # 't'*32, the key the k == 32 tables cannot hold
FORMATS = ("pairs", "split", "packed")


# ------------------------------------------------------------------ fixtures

@pytest.fixture(scope="module")
def eng():
    e = api.KmerCuda(0)
    yield e
    e.close()


class _OracleTables:
    """O.np_count of each (input, k) once; the three result formats of a call and later tests reuse it."""

    def __init__(self, keep=4):
        self.keep, self.tables = keep, {}

    def __call__(self, name, flat, off, k):
        key = (name, k)
        if key not in self.tables:
            if len(self.tables) >= self.keep:
                self.tables.pop(next(iter(self.tables)))
            self.tables[key] = O.np_count(flat, off, k)
        return self.tables[key]


@pytest.fixture(scope="module")
def oracle():
    return _OracleTables()


# ------------------------------------------------------------------ the branch and its launches (restated from api.cu)

def piece_bounds(n_bases):
    """[(b0, b1)] of the pieces the pipelined branch copies and partitions (submit_count_common, step 2)."""
    n_tiles = (n_bases + TILE - 1) // TILE
    n_pieces = 8 if n_tiles >= 8 else 1
    out = []
    for i in range(n_pieces):
        t0, t1 = n_tiles * i // n_pieces, n_tiles * (i + 1) // n_pieces
        out.append((t0 * TILE, min(n_bases, t1 * TILE)))
    return out


def branch(n_bases, n_rows, k):
    """('plain', 0) or ('pipelined', bucket groups): the plan has ceil(windows / 1200) buckets, counted in 8 groups from
    4096 buckets on (make_partition_plan, TARGET_KMERS_PER_BUCKET)."""
    if not (14 <= k <= 32 and n_rows and n_bases >= PIPELINE_MIN_BASES):
        return "plain", 0
    windows = max(n_bases - n_rows * (k - 1), 0)
    return "pipelined", 8 if -(-windows // 1200) >= 4096 else 1


def launch_range(n_bases, n_rows, k, fmt, recount=False):
    """(lo, hi) kernel launches of one host-buffer GROUP BY that succeeds.
    Both branches: status reset + rows_prepare, and resolve_bad_row at the end.
      plain, k <= 13:  dense count + compact;
      plain, k >= 14:  partition + bucket count, then tier 2's decide / clear / insert / compact;
      pipelined:       one partition per piece (8), one bucket count per group, tier 2's four kernels.
    The packed format adds one pack launch (plain) or one per group whose cursor moved (pipelined: none when no k-mer
    occurs once, e.g. every read twice); a tier-3 recount adds status reset + hash insert + compact, and then the plain
    download (one pack launch when packed)."""
    kind, groups = branch(n_bases, n_rows, k)
    if kind == "plain":
        n = 2 + (2 if k <= 13 else 2 + 4) + 1
        extra = (1, 1) if fmt == "packed" else (0, 0)
    else:
        n = 2 + 8 + groups + 4 + 1
        extra = (0, groups) if fmt == "packed" else (0, 0)
        if recount:
            n += 3
            extra = (1, groups + 1) if fmt == "packed" else (0, 0)
    return n + extra[0], n + extra[1]


# ------------------------------------------------------------------ inputs

def _mixed_case_acgt(rng, n):
    flat = datagen.DNA_CHARS[rng.integers(0, 4, size=n, dtype=np.uint8)]
    return flat | (rng.integers(0, 2, size=n, dtype=np.uint8) << 5).astype(np.uint8)


def _off_from_lens(lens):
    off = np.zeros(len(lens) + 1, np.uint64)
    off[1:] = np.cumsum(np.asarray(lens, np.int64)).astype(np.uint64)
    return off


def _poly_t(flat, off, rows):
    """Rows of 'T' / 't' only: at k == 32 their windows are the special key, at smaller k a long homopolymer."""
    flat = flat.copy()
    for i, r in enumerate(rows):
        flat[int(off[r]):int(off[r + 1])] = ord("T") if i % 2 == 0 else ord("t")
    return flat


def ragged_exact(seed, n_bases, min_len=100, max_len=1000):
    """Random mixed-case ragged rows of exactly n_bases bases, three of them poly-T."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(min_len, max_len + 1, size=2 * n_bases // min_len + 2)
    cs = np.cumsum(lens)
    j = int(np.searchsorted(cs, n_bases))
    lens = lens[: j + 1].copy()
    lens[-1] -= int(cs[j]) - n_bases
    if lens[-1] < min_len:
        lens[-2] += lens[-1]
        lens = lens[:-1]
    off = _off_from_lens(lens)
    flat = _poly_t(_mixed_case_acgt(rng, n_bases), off, [3, len(lens) // 2, len(lens) - 1])
    return flat, off


def _rows_from_cuts(cuts, n_bases, k, rng, whole=(), max_len=3000):
    """Row offsets with a row boundary at every cut; the gaps between cuts are filled with rows of k..max_len bases,
    except the gaps listed in `whole`, which stay one row."""
    pts = sorted(set([0, n_bases] + [int(c) for c in cuts]))
    off = [0]
    for a, b in zip(pts, pts[1:]):
        assert b - a >= k, (a, b)
        p = a
        if (a, b) not in whole:
            while b - p > max_len + k:
                p += int(rng.integers(k, max_len + 1))
                off.append(p)
        off.append(b)
    return np.array(off, np.uint64)


EDGE_N = 6_000_011
EDGE_ENDS = ("b1", "b1+1", "b1+k-1", "b1-1", "b1+63", "b1+64", "k|k")


def edge_columns(k):
    """Two columns of EDGE_N bases whose rows sit on the piece edges.
    'straddle': a row of exactly k bases across every inner piece boundary b1 but two, and one row longer than a piece
                across those two;
    'ends':     at each inner boundary rows end at one of b1, b1+1, b1+k-1, b1-1, b1+63, b1+64, or two rows of exactly
                k bases meet at b1 (rotated with k, so every k sees each case at some piece)."""
    rng = np.random.default_rng(1000 + k)
    b1s = [b1 for _, b1 in piece_bounds(EDGE_N)[:-1]]
    flat = _mixed_case_acgt(rng, EDGE_N)
    cuts = []
    for i, b in enumerate(b1s):
        if i in (2, 3):
            continue
        s = b - (1 + (5 * i) % (k - 1))          # k-row [s, s+k) crosses b with 1..k-1 bases before it
        cuts += [s, s + k]
    long_row = (b1s[2] - 2777, b1s[3] + 2555)
    assert long_row[1] - long_row[0] > max(b1 - b0 for b0, b1 in piece_bounds(EDGE_N))
    cuts += list(long_row)
    off_s = _rows_from_cuts(cuts, EDGE_N, k, rng, whole={long_row})
    cuts = []
    for i, b in enumerate(b1s):
        e = EDGE_ENDS[(i + k) % len(EDGE_ENDS)]
        cuts += {"b1": [b], "b1+1": [b + 1], "b1+k-1": [b + k - 1], "b1-1": [b - 1], "b1+63": [b + 63], "b1+64": [b + 64],
                 "k|k": [b - k, b, b + k]}[e]
    off_e = _rows_from_cuts(cuts, EDGE_N, k, rng)
    out = {}
    for name, off in (("straddle", off_s), ("ends", off_e)):
        lens = np.diff(off.astype(np.int64))
        rows_t = [int(i) for i in np.nonzero(lens >= 40)[0][[0, -1]]]
        out[name] = (_poly_t(flat, off, rows_t), off)
    return out


def tiny_rows(k, n_rows=1 << 19):
    """Half a million rows of k..k+3 bases (8 to 18 MB): nearly every base is near a row start."""
    rng = np.random.default_rng(77 + k)
    off = _off_from_lens(rng.integers(k, k + 4, size=n_rows))
    flat = _mixed_case_acgt(rng, int(off[-1]))
    flat[int(off[5]):int(off[9])] = ord("T")     # four poly-T rows
    return flat, off


def rows_input(rows):
    flat, off = O.rows_to_flat(rows)
    return np.frombuffer(flat, np.uint8), off


def _reads_as_rows(flat, off):
    return [bytes(flat[int(off[i]):int(off[i + 1])]).decode() for i in range(len(off) - 1)]


# ------------------------------------------------------------------ one call in every format, checked against the oracle

def sorted_table(keys, counts):
    o = np.argsort(keys, kind="stable")
    return keys[o], counts[o]


def _union(u, keys, counts):
    return sorted_table(np.concatenate([u, keys]), np.concatenate([np.ones(u.size, np.uint64), counts]))


def count_fmt(eng, fmt, flat, off, k):
    """(launches, table keys, table counts, n_kmers, checked extras) of one host-buffer GROUP BY in `fmt`."""
    before = eng.launches
    if fmt == "pairs":
        keys, counts, n = eng.count_kmers(flat, k, off)
        return eng.launches - before, keys, counts, n, None
    if fmt == "split":
        u, keys, counts, n = eng.count_kmers_split(flat, k, off)
        nb = 8
    else:
        u, keys, counts, n, nb = eng.count_kmers_packed(flat, k, off)
        assert nb == (2 * k + 7) // 8, (k, nb)
    launches = eng.launches - before
    su = np.sort(u)
    assert not (su[1:] == su[:-1]).any(), "a bare code came back twice"
    at = np.minimum(np.searchsorted(su, keys), max(su.size - 1, 0))
    assert su.size == 0 or not (su[at] == keys).any(), "a k-mer came back both bare and as a pair"
    uk, uc = _union(u, keys, counts)
    return launches, uk, uc, n, su


def check_formats(eng, flat, off, k, want, tag, recount=False, expect_branch=None):
    """All three formats equal the oracle table `want`; the launch count matches the branch the size selects, with
    (recount=True), without (False) or with or without (None) a tier-3 recount."""
    ok, oc, on = want
    n_bases, n_rows = int(off[-1]), len(off) - 1
    if expect_branch is not None:
        assert branch(n_bases, n_rows, k) == expect_branch, (tag, k)
    bare_split = None
    for fmt in FORMATS:
        launches, keys, counts, n, bare = count_fmt(eng, fmt, flat, off, k)
        if fmt == "pairs":
            keys, counts = sorted_table(keys, counts)
        assert n == on, (tag, k, fmt)
        assert np.array_equal(keys, ok) and np.array_equal(counts, oc), (tag, k, fmt)
        if k == 32 and ok.size and ok[-1] == SPECIAL:
            assert (keys == SPECIAL).sum() == 1 and counts[-1] == oc[-1], (tag, fmt, "the k == 32 key 't'*32")
        if fmt == "split":
            bare_split = bare
        elif fmt == "packed":
            assert np.array_equal(bare, bare_split), (tag, k, "packed bare codes != split bare codes")
        lo, hi = launch_range(n_bases, n_rows, k, fmt, bool(recount))
        if recount is None:                 # the input may or may not need the tier-3 recount
            hi = launch_range(n_bases, n_rows, k, fmt, True)[1]
        assert lo <= launches <= hi, (tag, k, fmt, launches, (lo, hi), branch(n_bases, n_rows, k))


# ------------------------------------------------------------------ A + B1: the branch each size takes; random ragged rows

SIZES = {"4MiB-1": (PIPELINE_MIN_BASES - 1, ("plain", 0)),
         "4MiB": (PIPELINE_MIN_BASES, ("pipelined", 1)),
         "6MB": (6_000_000, ("pipelined", 8))}


def test_launch_counts_pin_the_branch():
    """The restated launch counts of the three shapes (pairs / split exact, packed a range)."""
    assert launch_range(4 * MiB - 1, 8000, 21, "pairs") == (9, 9)
    assert launch_range(4 * MiB, 4096, 21, "split") == (16, 16)
    assert launch_range(4 * MiB, 4096, 21, "packed") == (16, 17)
    assert launch_range(6_000_000, 6000, 32, "pairs") == (23, 23)
    assert launch_range(6_000_000, 6000, 32, "packed") == (23, 31)
    assert launch_range(6_000_000, 6000, 13, "pairs") == (5, 5)
    assert [b for _, b in piece_bounds(4 * MiB)] == [(i + 1) * (MiB // 2) for i in range(8)]


@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("size", list(SIZES))
def test_ragged_sizes_all_formats(eng, oracle, size, k):
    n_bases, want_branch = SIZES[size]
    flat, off = ragged_exact(4000 + n_bases % 97, n_bases)
    assert int(off[-1]) == n_bases
    check_formats(eng, flat, off, k, oracle(size, flat, off, k), size, expect_branch=want_branch)


def test_dense_k13_stays_plain(eng, oracle):
    flat, off = datagen.synth_reads(13, 6000, 1000)
    check_formats(eng, flat, off, 13, oracle("k13reads", flat, off, 13), "k13", expect_branch=("plain", 0))


# ------------------------------------------------------------------ B2-B4: rows on the piece edges, tiny rows, odd sizes

@pytest.mark.parametrize("k", KS)
def test_rows_on_piece_edges(eng, k):
    for name, (flat, off) in edge_columns(k).items():
        assert int(off[-1]) == EDGE_N and branch(EDGE_N, len(off) - 1, k) == ("pipelined", 8)
        check_formats(eng, flat, off, k, O.np_count(flat, off, k), name)


@pytest.mark.parametrize("k", KS)
def test_a_million_tiny_rows(eng, k):
    flat, off = tiny_rows(k)
    assert branch(int(off[-1]), len(off) - 1, k)[0] == "pipelined"
    # a row of k..k+3 bases is at least one partition record: far more records per k-mer than the plan expects, so
    # the buckets overflow into the spill list and, at most k, past it into the recount
    check_formats(eng, flat, off, k, O.np_count(flat, off, k), "tiny rows", recount=None)


@pytest.mark.parametrize("k", KS)
def test_column_not_a_multiple_of_16(eng, k):
    n_bases = 5 * MiB + 7
    flat, off = ragged_exact(77, n_bases, 50, 2000)
    assert n_bases % 16 and branch(n_bases, len(off) - 1, k)[0] == "pipelined"
    check_formats(eng, flat, off, k, O.np_count(flat, off, k), "odd size")


# ------------------------------------------------------------------ C: tiers 2 and 3 through the pipelined branch

def _dev_count_tiers(eng, flat, off, k):
    """The device API on the same input and k (same plan): (n_tier2, n_overflow) it reports, and its table."""
    import torch
    d_seq = torch.from_numpy(np.concatenate([flat, np.zeros(64, np.uint8)])).cuda()
    d_off = torch.from_numpy(off.astype(np.int64)).cuda()
    cap = eng.max_kmers(int(off[-1]), len(off) - 1, k)
    d_pairs = torch.empty((cap, 2), dtype=torch.int64, device="cuda")
    eng.dev_count(d_seq, int(off[-1]), d_off, len(off) - 1, k, d_pairs, algo=api.ALGO_AUTO)
    r = eng.dev_finish()
    p = d_pairs[: r.n_distinct].cpu().numpy().view(np.uint64)
    return int(r.n_tier2), int(r.n_overflow), sorted_table(p[:, 0].copy(), p[:, 1].copy())


def tier2_doubled_reads():
    """Every read twice (test_leaf_table_full_goes_to_tier2): more repeated k-mers in a bucket than its leaf table holds."""
    rows = _reads_as_rows(*datagen.synth_reads(77, 3000, 1000))
    return rows_input(rows + rows)


def tier2_mixed_repeats():
    """Random reads with period-8 and period-2 repeats and long homopolymers (test_partition_tiers_mixed_input, scaled
    up to a pipelined size): the repeats' buckets spill."""
    rows = _reads_as_rows(*datagen.synth_reads(5, 5000, 1000))
    rep = ["ACGTTGCA" * 2500, "A" * 20000, "AC" * 10000, "t" * 12000]
    return rows_input(rows[:2500] + rep[:2] + rows[2500:] + rep[2:])


def tier3_homopolymers():
    """5 MB of homopolymer and short-period repeats: even the spill list overflows, the batch is recounted."""
    rows = _reads_as_rows(*datagen.synth_reads(5, 50, 1000))
    return rows_input(["T" * 3_000_000, "A" * 2_000_000, "AC" * 100_000, "GATTACA" * 20_000] + rows)


TIER_CASES = [("tier2_doubled_reads", tier2_doubled_reads, 2, (21, 31)),
              ("tier2_mixed_repeats", tier2_mixed_repeats, 2, (21, 32)),
              ("tier3_homopolymers", tier3_homopolymers, 3, (21, 32))]


@pytest.mark.parametrize("name,make,tier,ks", TIER_CASES, ids=[c[0] for c in TIER_CASES])
def test_tiers_through_the_pipeline(eng, name, make, tier, ks):
    flat, off = make()
    assert int(off[-1]) >= PIPELINE_MIN_BASES
    for k in ks:
        want = O.np_count(flat, off, k)
        n_tier2, n_overflow, (dk, dc) = _dev_count_tiers(eng, flat, off, k)
        print(f"{name} k={k}: n_bases={int(off[-1])} rows={len(off) - 1} device API n_tier2={n_tier2} n_overflow={n_overflow}")
        # the precondition: this input and k reach the tier under test (never weakened: resize the input instead)
        if tier == 2:
            assert n_tier2 > 0 and n_overflow == 0, (name, k, n_tier2, n_overflow)
        else:
            assert n_overflow > 0, (name, k, n_tier2, n_overflow)
        assert np.array_equal(dk, want[0]) and np.array_equal(dc, want[1]), (name, k, "device API")
        check_formats(eng, flat, off, k, want, name, recount=tier == 3)


# ------------------------------------------------------------------ D: input errors through the pipelined branch

ERRORS = {O.ORC_INVALID_DNA: (api.KMER_ERR_INVALID_DNA, "22P02", "Invalid DNA Sequence",
                              "Valid characters are A, C, G, T (case-insensitive)."),
          O.ORC_INVALID_K: (api.KMER_ERR_INVALID_K, "22023", "Invalid KMER Length", "")}


def expect_reference_error(eng, flat, off, k, tag):
    """Every format raises what the reference raises first: status, SQLSTATE, message, detail and row."""
    with pytest.raises(O.OracleError) as oe:
        O.np_generate(flat, off, k)
    want = ERRORS[oe.value.code] + (oe.value.row,)
    for call in (eng.count_kmers, eng.count_kmers_split, eng.count_kmers_packed):
        with pytest.raises(api.KmerSqlError) as ei:
            call(flat, k, off)
        e = ei.value
        assert (e.status, e.sqlstate, e.message, e.detail, e.row) == want, (tag, k, call.__name__)
    return want


@pytest.mark.parametrize("k", (21, 32))
def test_invalid_bytes_at_piece_edges(eng, oracle, k):
    flat, off = ragged_exact(4000 + 6_000_000 % 97, 6_000_000)
    n = int(off[-1])
    assert branch(n, len(off) - 1, k) == ("pipelined", 8)
    bounds = piece_bounds(n)
    where = [0, n - 1]
    for i in (0, 3, 6):
        b1 = bounds[i][1]
        where += [b1 - 1, b1, b1 + k - 2, b1 + 63, b1 + 64]
    for pos in where:
        for bad in (ord("N"), 0x00, 0x80 | ord("a")):
            f2 = flat.copy()
            f2[pos] = bad
            st = expect_reference_error(eng, f2, off, k, (pos, bad))
            assert st[0] == api.KMER_ERR_INVALID_DNA
    # the context is still good: the same column without the bad byte
    check_formats(eng, flat, off, k, oracle("6MB", flat, off, k), "after errors")


@pytest.mark.parametrize("k", (21, 32))
def test_short_rows_and_precedence(eng, k):
    flat, off = ragged_exact(4000 + 6_000_000 % 97, 6_000_000)
    n = int(off[-1])
    b1 = piece_bounds(n)[4][1]
    r = int(np.searchsorted(off, b1, side="right")) - 1        # the row across piece 4's end
    short = np.insert(off, r + 1, off[r] + np.uint64(k - 1))     # row r becomes k-1 bases, the rest is row r+1
    assert np.diff(short.astype(np.int64)).min() == k - 1 and int(short[-1]) == n
    assert expect_reference_error(eng, flat, short, k, "short row")[::4] == (api.KMER_ERR_INVALID_K, r)
    # an invalid byte in a later row: the short row is reported
    f2 = flat.copy()
    f2[int(short[r + 3]) + 5] = ord("N")
    assert expect_reference_error(eng, f2, short, k, "short, then bad")[::4] == (api.KMER_ERR_INVALID_K, r)
    # an invalid byte in an earlier row: that row is reported
    f2 = flat.copy()
    f2[int(short[r - 2]) + 5] = ord("N")
    assert expect_reference_error(eng, f2, short, k, "bad, then short")[::4] == (api.KMER_ERR_INVALID_DNA, r - 2)
    # both in the same row: dna_in runs before generate_kmers
    f2 = flat.copy()
    f2[int(short[r]) + 1] = 0x00
    assert expect_reference_error(eng, f2, short, k, "bad in the short row")[::4] == (api.KMER_ERR_INVALID_DNA, r)


# ------------------------------------------------------------------ E: one context through a sequence of calls

def _expect_table(got, want, tag):
    keys, counts, n = got
    keys, counts = sorted_table(keys, counts)
    assert n == want[2] and np.array_equal(keys, want[0]) and np.array_equal(counts, want[1]), tag


def _split_table(got):
    u, keys, counts, n = got[:4]
    return (*_union(u, keys, counts), n)


def test_one_context_many_calls(oracle):
    e = api.KmerCuda(0)
    try:
        big, big_off = ragged_exact(4000 + 6_000_000 % 97, 6_000_000)
        mid, mid_off = datagen.synth_reads(60, 4096, 1024)
        small, small_off = datagen.synth_ragged(61, 2000, 500, min_len=40, mixed_case=True)
        t3, t3_off = tier3_homopolymers()
        # 1. pipelined success
        _expect_table(e.count_kmers(big, 21, big_off), oracle("6MB", big, big_off, 21), "1: pipelined")
        # 2. pipelined error
        bad = big.copy()
        bad[piece_bounds(6_000_000)[2][1] + 3] = ord("N")
        with pytest.raises(api.KmerSqlError) as ei:
            e.count_kmers_split(bad, 21, big_off)
        assert ei.value.status == api.KMER_ERR_INVALID_DNA
        # 3. pipelined success
        _expect_table(_split_table(e.count_kmers_split(big, 31, big_off)), oracle("6MB", big, big_off, 31), "3: after an error")
        # 4. tier 3
        _expect_table(e.count_kmers(t3, 21, t3_off), O.np_count(t3, t3_off, 21), "4: tier 3")
        # 5. packed, 6. pairs
        _expect_table(_split_table(e.count_kmers_packed(big, 27, big_off)), oracle("6MB", big, big_off, 27), "5: packed")
        _expect_table(e.count_kmers(mid, 32, mid_off), O.np_count(mid, mid_off, 32), "6: pairs, k = 32")
        # 7. a smaller call, then a larger one
        _expect_table(_split_table(e.count_kmers_split(small, 21, small_off)), O.np_count(small, small_off, 21), "7: small")
        tiny, tiny_off = tiny_rows(14)
        _expect_table(e.count_kmers(tiny, 14, tiny_off), O.np_count(tiny, tiny_off, 14), "7: larger")
        # stale padding: an 'N' at p >= 4 MiB fails the call; cut at n_bases = p, it lies behind the column in the
        # workspace the context reuses and must not be seen
        j = int(np.nonzero((big_off > 4 * MiB + 5000) & (big_off % 16 != 0))[0][0])
        p = int(big_off[j])
        bad = big.copy()
        bad[p] = ord("N")
        with pytest.raises(api.KmerSqlError) as ei:
            e.count_kmers(bad, 21, big_off)
        assert (ei.value.status, ei.value.row) == (api.KMER_ERR_INVALID_DNA, j)
        cut, cut_off = bad[:p], big_off[: j + 1]
        want = O.np_count(cut, cut_off, 21)
        assert branch(p, j, 21)[0] == "pipelined"
        _expect_table(e.count_kmers(cut, 21, cut_off), want, "stale 'N' past n_bases: pairs")
        _expect_table(_split_table(e.count_kmers_split(cut, 21, cut_off)), want, "stale 'N' past n_bases: split")
        _expect_table(_split_table(e.count_kmers_packed(cut, 21, cut_off)), want, "stale 'N' past n_bases: packed")
    finally:
        e.close()


# ------------------------------------------------------------------ F: the output-capacity contract of the device API

SENTINEL = 0x5A5A5A5A5A5A5A5A
SLACK = 256


def _out(n, width):
    """A view of n rows (capacity n) at the front of an allocation whose rest holds a sentinel pattern."""
    import torch
    base = torch.full((n + SLACK, width) if width > 1 else (n + SLACK,), SENTINEL, dtype=torch.int64, device="cuda")
    return base, base[:n]


def _untouched(base, n):
    return bool((base[n:] == SENTINEL).all())


def _dev(flat, off):
    import torch
    return (torch.from_numpy(np.concatenate([flat, np.zeros(64, np.uint8)])).cuda(),
            torch.from_numpy(off.astype(np.int64)).cuda())


def _pairs_of(view, r):
    p = view[: r.n_distinct].cpu().numpy().view(np.uint64)
    return sorted_table(p[:, 0].copy(), p[:, 1].copy())


def capacity_case(eng, n, run, check, width=2, tag=""):
    """Capacity n succeeds and is exact, n - 1 raises KMER_ERR_CAPACITY; neither writes past its view; the next call on
    the same context with room is exact again."""
    assert n >= 1, tag
    base, view = _out(n, width)
    run(view)
    check(view, eng.dev_finish())
    assert _untouched(base, n), (tag, "exact capacity: wrote past the view")
    base, view = _out(n - 1, width)
    run(view)
    with pytest.raises(api.KmerSqlError) as ei:
        eng.dev_finish()
    assert (ei.value.status, ei.value.sqlstate) == (api.KMER_ERR_CAPACITY, "XX000"), tag
    assert ei.value.message == "kmer_cuda: output buffer too small", tag
    assert _untouched(base, n - 1), (tag, "one short: wrote past the view")
    base, view = _out(n + 100, width)
    run(view)
    check(view, eng.dev_finish())
    assert _untouched(base, n + 100), tag


def _capacity_input(k):
    """Random ragged rows, a tenth of them twice (groups with count > 1), and poly-T rows."""
    flat, off = datagen.synth_ragged(700 + k, 2500, 400, min_len=40, mixed_case=True)
    rows = _reads_as_rows(flat, off)
    return rows_input(rows + rows[::10] + ["T" * 100, "t" * 40])


@pytest.mark.parametrize("k,algo", [(9, api.ALGO_DENSE), (21, api.ALGO_HASH), (21, api.ALGO_PARTITION), (21, api.ALGO_TWO_PASS),
                                    (32, api.ALGO_HASH), (32, api.ALGO_PARTITION), (32, api.ALGO_TWO_PASS)])
def test_capacity_dev_count(eng, k, algo):
    """At k = 32 the key 't'*32 is appended after every other group: one slot short, it is the one without room."""
    flat, off = _capacity_input(k)
    ok, oc, on = O.np_count(flat, off, k)
    if k == 32:
        assert ok[-1] == SPECIAL and oc[-1] > 1
    d_seq, d_off = _dev(flat, off)

    def run(view):
        eng.dev_count(d_seq, int(off[-1]), d_off, len(off) - 1, k, view, algo=algo)

    def check(view, r):
        keys, counts = _pairs_of(view, r)
        assert r.n_kmers == on and np.array_equal(keys, ok) and np.array_equal(counts, oc), (k, algo)

    capacity_case(eng, ok.size, run, check, tag=(k, algo))


def test_capacity_dev_count_split(eng):
    k = 21
    flat, off = _capacity_input(k)
    ok, oc, on = O.np_count(flat, off, k)
    d_seq, d_off = _dev(flat, off)
    n_bases, n_rows = int(off[-1]), len(off) - 1
    _, uq = _out(ok.size, 1)
    _, pr = _out(ok.size, 2)
    eng.dev_count_split(d_seq, n_bases, d_off, n_rows, k, uq, pr)
    r = eng.dev_finish()
    nu, nd = int(r.n_unique), int(r.n_distinct)
    assert nu > 0 and nd > 0 and nu + nd == ok.size

    def check(u_view, p_view, r):
        assert (r.n_unique, r.n_distinct, r.n_kmers) == (nu, nd, on)
        u = u_view[:nu].cpu().numpy().view(np.uint64)
        keys, counts = _pairs_of(p_view, r)
        uk, uc = _union(u, keys, counts)
        assert np.intersect1d(u, keys).size == 0 and np.array_equal(uk, ok) and np.array_equal(uc, oc)

    for u_cap, p_cap, fits in ((nu, nd, True), (nu - 1, nd, False), (nu, nd - 1, False), (nu + 50, nd + 50, True)):
        ub, uv = _out(u_cap, 1)
        pb, pv = _out(p_cap, 2)
        eng.dev_count_split(d_seq, n_bases, d_off, n_rows, k, uv, pv)
        if fits:
            check(uv, pv, eng.dev_finish())
        else:
            with pytest.raises(api.KmerSqlError) as ei:
                eng.dev_finish()
            assert (ei.value.status, ei.value.sqlstate) == (api.KMER_ERR_CAPACITY, "XX000"), (u_cap, p_cap)
        assert _untouched(ub, u_cap) and _untouched(pb, p_cap), (u_cap, p_cap)


def test_capacity_dev_extract(eng):
    k = 17
    flat, off = _capacity_input(k)
    want = O.np_generate(flat, off, k)
    d_seq, d_off = _dev(flat, off)

    def run(view):
        eng.dev_extract(d_seq, int(off[-1]), d_off, len(off) - 1, k, view)

    def check(view, r):
        assert r.n_kmers == want.size and np.array_equal(view.cpu().numpy().view(np.uint64)[: want.size], want)

    capacity_case(eng, want.size, run, check, width=1, tag="extract")


def test_capacity_dev_shard_count(eng):
    """Two simulated ranks (the slicing of test_sharded_count_simulated_ranks); owner 0's table at its exact size."""
    import torch
    G, k = 2, 21
    shards = [datagen.synth_ragged(500 + 10 * G + r, 1500, 300, min_len=40, mixed_case=(r % 2 == 1)) for r in range(G)]
    total = sum(eng.max_kmers(int(o[-1]), len(o) - 1, k) for _, o in shards)
    plan = eng.shard_plan(total, k, G)
    send_recs, send_fill = [], []
    for flat, off in shards:
        d_seq, d_off = _dev(flat, off)
        recs = torch.empty(plan.recs_bytes_per_peer * G, dtype=torch.uint8, device="cuda")
        fill = torch.empty(plan.buckets_per_rank * G, dtype=torch.int64, device="cuda")
        eng.dev_shard_partition(d_seq, int(off[-1]), d_off, len(off) - 1, plan, recs, fill)
        eng.dev_finish()
        send_recs.append(recs)
        send_fill.append(fill)
    rb, fb = plan.recs_bytes_per_peer, plan.buckets_per_rank
    owner = 0
    recv_recs = torch.cat([send_recs[r][owner * rb:(owner + 1) * rb] for r in range(G)])
    recv_fill = torch.cat([send_fill[r][owner * fb:(owner + 1) * fb] for r in range(G)])
    _, pairs = _out(total, 2)
    eng.dev_shard_count(plan, recv_recs, recv_fill, pairs)
    r0 = eng.dev_finish()
    want = _pairs_of(pairs, r0)
    # the owner's share of the oracle table: the union over both owners is checked by test_gpu_parity
    flat = np.concatenate([s[0] for s in shards])
    offs = np.concatenate([shards[0][1], shards[1][1][1:] + shards[0][1][-1]])
    ok, oc, on = O.np_count(flat, offs, k)
    idx = np.searchsorted(ok, want[0])
    assert (idx < ok.size).all() and np.array_equal(ok[idx], want[0]) and np.array_equal(oc[idx], want[1])

    def run(view):
        eng.dev_shard_count(plan, recv_recs, recv_fill, view)

    def check(view, r):
        keys, counts = _pairs_of(view, r)
        assert r.n_kmers == r0.n_kmers and np.array_equal(keys, want[0]) and np.array_equal(counts, want[1])

    capacity_case(eng, int(r0.n_distinct), run, check, tag="shard count")


def test_capacity_dev_dense_emit(eng):
    import torch
    k, G, rank = 7, 4, 1
    flat, off = datagen.synth_ragged(901, 300, 200, min_len=16)
    ok, oc, on = O.np_count(flat, off, k)
    d_seq, d_off = _dev(flat, off)
    table = torch.empty(4 ** k, dtype=torch.int64, device="cuda")
    eng.dev_dense_table(d_seq, int(off[-1]), d_off, len(off) - 1, k, table)
    eng.dev_finish()
    mine = ok % np.uint64(G) == np.uint64(rank)
    assert 0 < mine.sum() < ok.size

    def run(view):
        eng.dev_dense_emit(table, k, rank, G, view)

    def check(view, r):
        keys, counts = _pairs_of(view, r)
        assert np.array_equal(keys, ok[mine]) and np.array_equal(counts, oc[mine])

    capacity_case(eng, int(mine.sum()), run, check, tag="dense emit")


def _pair_table(flat, off, k):
    import torch
    ok, oc, on = O.np_count(flat, off, k)
    t = torch.from_numpy(np.stack([ok, oc], axis=1).view(np.int64)).cuda()
    return ok, oc, t


@pytest.mark.parametrize("k", (21, 32))
def test_capacity_dev_merge_emit(eng, k):
    """Two halves of one table merged; at k = 32 the key 't'*32 goes through the merge too."""
    ok, oc, t = _pair_table(*_capacity_input(k), k)
    if k == 32:
        assert ok[-1] == SPECIAL
    half = ok.size // 2

    def run(view):
        eng.dev_merge_begin(ok.size)
        eng.dev_merge_add(t[half:], ok.size - half, 0, 1)
        eng.dev_merge_add(t[:half], half, 0, 1)
        eng.dev_merge_emit(k, view)

    def check(view, r):
        keys, counts = _pairs_of(view, r)
        assert r.n_distinct == ok.size and np.array_equal(keys, ok) and np.array_equal(counts, oc)

    capacity_case(eng, ok.size, run, check, tag=("merge", k))


def test_merge_table_full(eng):
    """merge_begin(1) has 1024 slots: 2000 distinct groups cannot all be placed."""
    ok, oc, t = _pair_table(*datagen.synth_reads(31, 20, 300), 21)
    assert ok.size > 2000
    t = t[:2000]
    base, view = _out(4000, 2)
    eng.dev_merge_begin(1)
    eng.dev_merge_add(t, 2000, 0, 1)
    eng.dev_merge_emit(21, view)
    with pytest.raises(api.KmerSqlError) as ei:
        eng.dev_finish()
    assert (ei.value.status, ei.value.sqlstate) == (api.KMER_ERR_CAPACITY, "XX000")
    assert ei.value.message == "kmer_cuda: merge table full (max_groups too small)"
    assert _untouched(base, 4000)
    # the same context with room
    eng.dev_merge_begin(2000)
    eng.dev_merge_add(t, 2000, 0, 1)
    eng.dev_merge_emit(21, view)
    r = eng.dev_finish()
    keys, counts = _pairs_of(view, r)
    assert np.array_equal(keys, ok[:2000]) and np.array_equal(counts, oc[:2000])
