"""The closed-form GROUP BY of genome-sampled reads (tests/coverage_util.py) against the general oracles (CPU only).

tests/test_coverage_gpu.py compares the GPU counter with coverage_table at sizes where sorting every window is not
practical, so coverage_table itself is pinned here: equal to O.np_count and to the C oracle's count, and its checksum equal
to the C oracle's multiset checksum of the rows, for every record width of the kernels' k range, without errors, at 0.2 %
and 2 % substitutions, for fixed and ragged reads.  Every input has reads at both ends of the genome, a poly-T run of 320
bases (count far above the coverage; the all-ones code at k = 32), a poly-A run, a (CA)n microsatellite, a copied segment
and two substitutions closer than k in one read.
"""
import numpy as np
import pytest

import coverage_util as CU
from oracle import oracle as O

KS = [14, 21, 26, 27, 31, 32]
ERRS = [0.0, 0.002, 0.02]


def _input(k, err, ragged):
    seed = 100 * k + int(err * 1000) * 2 + int(ragged)
    (flat, off), (genome, starts, err_pos) = CU.sample_reads(seed, 24_000, 1600, 300, err, ragged=ragged)
    return flat, off, genome, starts, err_pos


@pytest.mark.parametrize("ragged", [False, True], ids=["fixed", "ragged"])
@pytest.mark.parametrize("err", ERRS, ids=[f"err{e}" for e in ERRS])
@pytest.mark.parametrize("k", KS)
def test_coverage_table_equals_the_oracles(corc, k, err, ragged):
    flat, off, genome, starts, err_pos = _input(k, err, ragged)
    lens = np.diff(off.astype(np.int64))
    keys, counts, n = CU.coverage_table(genome, starts, lens, err_pos, flat, k)
    ok, oc, on = O.np_count(flat, off, k)
    assert n == on and np.array_equal(keys, ok) and np.array_equal(counts, oc)
    ck, cc, cn = corc.count(flat, off, k)
    o = np.argsort(ck, kind="stable")
    assert cn == n and np.array_equal(ck[o], keys) and np.array_equal(cc[o], counts)
    s, sn = corc.multiset_checksum(flat, off, k)
    assert sn == n and O.np_table_checksum(keys, counts) == s
    # the input reaches what it is built to reach
    assert int(counts.sum()) == n
    poly_t = (1 << (2 * k)) - 1
    assert counts[np.searchsorted(keys, np.uint64(poly_t))] > 10 * counts.mean()
    if err:
        assert np.count_nonzero(np.diff(err_pos) < k) > 0


def test_reads_touch_both_genome_ends_and_keep_their_case():
    (flat, off), (genome, starts, err_pos) = CU.sample_reads(5, 10_000, 50, 200, 0.0, ragged=True)
    lens = np.diff(off.astype(np.int64))
    assert starts[0] == 0 and starts[-1] + lens[-1] == genome.size
    assert (starts >= 0).all() and (starts + lens <= genome.size).all()
    for r in range(lens.size):
        row = flat[int(off[r]):int(off[r + 1])]
        assert (row >= ord("a")).all() or (row < ord("a")).all()
        assert np.array_equal(O._CODE_LUT[row], genome[starts[r]:starts[r] + lens[r]])


def test_error_windows_are_the_windows_that_differ_from_the_genome():
    """Every window of a mutated read that differs from its genome window is an error window, and each is listed once;
    a window that covers a substitution always differs, since a substitution changes the base."""
    k = 21
    (flat, off), (genome, starts, err_pos) = CU.sample_reads(8, 12_000, 400, 120, 0.03, ragged=True)
    lens = np.diff(off.astype(np.int64))
    wid = CU.error_windows(lens, err_pos, k)
    assert np.array_equal(wid, np.unique(wid))
    offs = off.astype(np.int64)
    differ = []
    c2 = O._CODE_LUT[flat]
    for r in range(lens.size):
        g = genome[starts[r]:starts[r] + lens[r]]
        bad = np.flatnonzero(c2[offs[r]:offs[r + 1]] != g)
        for o in range(lens[r] - k + 1):
            if bad.size and ((bad >= o) & (bad < o + k)).any():
                differ.append(offs[r] + o)
    assert np.array_equal(wid, np.array(differ, np.int64))


def test_group_sum_is_exact_beyond_float_precision():
    keys = np.array([5, 3, 5, 3, 9], np.uint64)
    counts = np.array([2 ** 53 + 1, 1, 2 ** 53, 2, 7], np.int64)
    k, c = CU.group_sum(keys, counts)
    assert k.tolist() == [3, 5, 9] and c.tolist() == [3, 2 ** 54 + 1, 7]
