"""Oracles of canonical counting: a k-mer and its reverse complement (a<->t, c<->g, order reversed) are one group, keyed by
canon(x) = min(x, rc(x)) -- on codes and, equally, on lower-case text.

Three independent restatements, pinned to each other by tests/test_canonical_oracle.py:
  * text_count: a Counter over min(s, rc(s)) of every window's lower-case text;
  * np_canonical_count: numpy, the canonical codes of O.np_generate's windows;
  * fold: a strand-specific table (any oracle's, or the GPU's) folded: count_canon(c) = count(c) + count(rc c) for c != rc c,
    count(c) for a palindrome.
and, for reads sampled from BOTH strands of a genome with errors, both_strands(): the strand-specific closed form of
tests/coverage_util.py folded.  That is exact because reverse-complementing a row maps every window to its reverse complement,
which has the same canonical code: the canonical table does not depend on which strand a read came from.
"""
from collections import Counter

import numpy as np

import coverage_util as CU
from kmer_extension_b200 import api
from oracle import oracle as O

_RC_TEXT = str.maketrans("acgt", "tgca")
COMP_ASCII = np.arange(256, dtype=np.uint8)
for _a, _b in zip(b"ACGTacgt", b"TGCAtgca"):
    COMP_ASCII[_a] = _b


def rc_text(s: str) -> str:
    return s.lower()[::-1].translate(_RC_TEXT)


def canon_text(s: str) -> str:
    s = s.lower()
    return min(s, rc_text(s))


def text_count(rows, k):
    """Counter {canonical lower-case text: count} over every window of every row (rows: str)."""
    c = Counter()
    for r in rows:
        for i in range(len(r) - k + 1):
            c[canon_text(r[i:i + k])] += 1
    return c


def np_canonical_count(flat, off, k):
    """(sorted distinct canonical codes, counts, n_windows), the triple of O.np_count."""
    codes = api.canonical_codes(O.np_generate(flat, off, k), k)
    keys, counts = np.unique(codes, return_counts=True)
    return keys.astype(np.uint64), counts.astype(np.uint64), int(codes.size)


def fold(keys, counts, k):
    """A strand-specific (keys, counts) table -> its canonical table (sorted keys, summed counts)."""
    keys = np.asarray(keys, np.uint64)
    return CU.group_sum(api.canonical_codes(keys, k), np.asarray(counts, np.int64))


def counter_of(keys, counts, k):
    """codes -> Counter of their text (for comparing with text_count)."""
    text = O.np_decode(np.asarray(keys, np.uint64), k) if len(keys) else np.zeros((0, k), np.uint8)
    return Counter({bytes(t).decode(): int(c) for t, c in zip(text, counts)})


def revcomp_rows(flat, off, which):
    """flat with the rows where which[r] is true reverse-complemented in place of themselves (case kept per base)."""
    flat = np.array(flat, np.uint8, copy=True)
    off = np.asarray(off, np.int64)
    rows = np.flatnonzero(which)
    if rows.size:
        lens = off[rows + 1] - off[rows]
        first = np.zeros(rows.size, np.int64)
        np.cumsum(lens[:-1], out=first[1:])
        rep = np.repeat(np.arange(rows.size), lens)
        i = np.arange(int(lens.sum())) - first[rep]                     # position inside the row
        dst = off[rows][rep] + i
        src = off[rows + 1][rep] - 1 - i
        flat[dst] = COMP_ASCII[flat[src]]
    return flat


def both_strands(seed, genome_len, n_reads, read_len, k, err_rate=0.0, ragged=False):
    """Reads of a seeded genome, about half of them from the reverse strand -> ((flat, off), canonical table triple)."""
    (flat, off), (genome, starts, err) = CU.sample_reads(seed, genome_len, n_reads, read_len, err_rate, ragged)
    keys, counts, n = CU.coverage_table(genome, starts, np.diff(off.astype(np.int64)), err, flat, k)
    ck, cc = fold(keys, counts, k)
    which = np.random.default_rng(seed + 1).integers(0, 2, len(off) - 1).astype(bool)
    return (revcomp_rows(flat, off, which), off), (ck, cc, n)
