"""Sequencing reads sampled from a known genome, and their exact GROUP BY kmer / count(*) in closed form.

Real input to the count is reads drawn from one genome at some coverage, with a few substitution errors: many k-mers occur
about `coverage` times, and a long tail of error k-mers occurs once.  `sample_reads` draws such a table (seeded), and
`coverage_table` computes its GROUP BY table from the genome, the read starts and the error positions, without sorting
every window: O(genome + error windows) plus one sort of about genome-many codes.  tests/test_coverage_oracle.py pins it
to O.np_count and the C oracle.

Why the closed form is exact: read r is genome[s_r : s_r + L_r] with substitutions at known offsets.  A window (r, o) that
covers no substitution equals genome window s_r + o; a window that covers one counts once under the code of the mutated
read.  So the count of genome window p is the number of reads whose windows reach p, less the error windows that map to
p; the table is the group-by-sum of (genome window codes, those counts) and (error window codes, 1).  Genome-level
repeats and error k-mers that equal a genome k-mer are merged by that group-by.
"""
import numpy as np

from oracle import oracle as O

UPPER_LOWER = np.frombuffer(b"ACGTacgt", np.uint8)
MIN_GENOME = 8192


def _genome(rng, G):
    """i.i.d. bases with a poly-T run (320 b), a poly-A run (200 b), a (CA)n microsatellite (300 b) and one segment of
    G/16 bases copied to a second place (a genome-level repeat)."""
    assert G >= MIN_GENOME
    g = rng.integers(0, 4, G, dtype=np.uint8)
    g[G // 8:G // 8 + 320] = 3
    g[3 * G // 8:3 * G // 8 + 200] = 0
    g[5 * G // 8:5 * G // 8 + 300] = np.tile(np.array([1, 0], np.uint8), 150)
    seg = G // 16
    g[7 * G // 8:7 * G // 8 + seg] = g[G // 4:G // 4 + seg]
    return g


def sample_reads(seed, genome_len, n_reads, read_len, err_rate=0.0, ragged=False, min_len=40):
    """Reads of a seeded genome -> ((flat ASCII uint8, off uint64[n+1]), (genome 2-bit uint8, starts int64, err_pos int64)).

    Read lengths are read_len, or uniform in [min_len, read_len] if ragged.  Starts are uniform over the genome; the first
    read starts at the genome's first base and the last read ends at its last base.  Every base is substituted with
    probability about err_rate (positions drawn with replacement, then deduplicated: cheap at 1e9 bases), and with
    err_rate > 0 read 1 always has two substitutions 5 bases apart.  Each read is upper or lower case.  err_pos are
    sorted positions in flat."""
    rng = np.random.default_rng(seed)
    G = int(genome_len)
    genome = _genome(rng, G)
    assert min_len <= read_len <= G and n_reads >= 2
    lens = rng.integers(min_len, read_len + 1, n_reads) if ragged else np.full(n_reads, read_len, np.int64)
    lens = lens.astype(np.int64)
    starts = rng.integers(0, G - lens + 1).astype(np.int64)
    starts[0], starts[-1] = 0, G - lens[-1]
    upper = rng.integers(0, 2, n_reads).astype(np.uint8)
    off = np.zeros(n_reads + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    N = int(off[-1])
    flat = np.empty(N, np.uint8)
    step = max(1, (32 << 20) // int(read_len))                       # about 32 M bases per block
    for r0 in range(0, n_reads, step):
        r1 = min(n_reads, r0 + step)
        b0, b1 = int(off[r0]), int(off[r1])
        src = np.repeat(starts[r0:r1] - off[r0:r1], lens[r0:r1]) + np.arange(b0, b1)
        flat[b0:b1] = UPPER_LOWER[np.repeat(upper[r0:r1] ^ 1, lens[r0:r1]) * 4 + genome[src]]
    err = np.zeros(0, np.int64)
    if err_rate > 0:
        err = rng.integers(0, N, rng.binomial(N, err_rate))
        err = np.unique(np.concatenate([err, off[1] + np.array([10, 15])]))
        old = O._CODE_LUT[flat[err]]
        lower = (flat[err] >= ord("a")).astype(np.uint8)
        flat[err] = UPPER_LOWER[lower * 4 + (old + rng.integers(1, 4, err.size).astype(np.uint8)) % 4]
    return (flat, off.astype(np.uint64)), (genome, starts, err)


def _codes_at(codes2, pos, k):
    """codes of the k-mers of a 2-bit array starting at positions pos"""
    acc = np.zeros(pos.size, np.uint64)
    for j in range(k):
        acc <<= np.uint64(2)
        acc |= codes2[pos + j]
    return acc


def error_windows(lens, err_pos, k):
    """Windows that cover at least one substitution, each once: sorted global window starts (positions in flat)."""
    lens = np.asarray(lens, np.int64)
    off = np.zeros(lens.size + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    err_pos = np.asarray(err_pos, np.int64)
    if err_pos.size == 0:
        return np.zeros(0, np.int64)
    r = np.searchsorted(off, err_pos, side="right") - 1
    e = err_pos - off[r]
    lo = np.maximum(e - k + 1, 0)
    hi = np.minimum(e, lens[r] - k)
    # err_pos is sorted, so inside a read hi never decreases: clipping lo behind the previous hi makes the ranges disjoint
    same = np.zeros(r.size, bool)
    same[1:] = r[1:] == r[:-1]
    prev_hi = np.empty_like(hi)
    prev_hi[0] = -1
    prev_hi[1:] = hi[:-1]
    lo = np.where(same, np.maximum(lo, prev_hi + 1), lo)
    n = np.maximum(hi - lo + 1, 0)
    first = np.zeros(n.size, np.int64)
    np.cumsum(n[:-1], out=first[1:])
    rep = np.repeat(np.arange(n.size), n)
    return off[r][rep] + lo[rep] + (np.arange(int(n.sum())) - first[rep])


def group_sum(keys, counts):
    """(keys, counts) with repeated keys -> sorted distinct keys and the int64 sums of their counts."""
    o = np.argsort(keys, kind="stable")
    sk, sc = keys[o], counts[o]
    if sk.size == 0:
        return sk.astype(np.uint64), sc.astype(np.uint64)
    head = np.flatnonzero(np.concatenate([[True], sk[1:] != sk[:-1]]))
    return sk[head].astype(np.uint64), np.add.reduceat(sc, head).astype(np.uint64)


def coverage_table(genome, starts, lens, err_pos, mutated_flat, k):
    """GROUP BY kmer / count(*) over the windows of the sampled reads -> (sorted distinct codes, counts, n_windows),
    the same triple as O.np_count."""
    genome = np.asarray(genome, np.uint8)
    starts = np.asarray(starts, np.int64)
    lens = np.asarray(lens, np.int64)
    G = genome.size
    W = G - k + 1
    gcodes = np.zeros(W, np.uint64)
    for j in range(k):
        gcodes <<= np.uint64(2)
        gcodes |= genome[j:W + j]
    v = lens >= k
    cnt = np.cumsum(np.bincount(starts[v], minlength=W + 1) - np.bincount(starts[v] + lens[v] - k + 1, minlength=W + 1))[:W]
    wid = error_windows(lens, err_pos, k)
    off = np.zeros(lens.size + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    r = np.searchsorted(off, wid, side="right") - 1
    cnt -= np.bincount(starts[r] + (wid - off[r]), minlength=W)
    assert (cnt >= 0).all()
    ecodes = _codes_at(O._CODE_LUT[np.asarray(mutated_flat, np.uint8)], wid, k) if wid.size else np.zeros(0, np.uint64)
    keep = cnt > 0
    keys, counts = group_sum(np.concatenate([gcodes[keep], ecodes]), np.concatenate([cnt[keep], np.ones(wid.size, np.int64)]))
    return keys, counts, int(np.maximum(lens - k + 1, 0).sum())


def reads_for(genome_len, coverage, read_len):
    """number of reads of length read_len that cover a genome of genome_len bases coverage times"""
    return max(2, int(round(genome_len * coverage / read_len)))
