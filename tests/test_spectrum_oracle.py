"""CPU tests of the abundance spectrum (count of counts): the numpy restatement the GPU tests compare with (tests/spectrum_util.py),
api.spectrum_rows (the SQL relation), and the argument checks of the four spectrum entry points, which need no device."""
import collections
import ctypes as C

import numpy as np
import pytest

import coverage_util as CU
import spectrum_util as S
from kmer_extension_b200 import api, datagen
from oracle import oracle as O


def _counter_spectrum(flat, off, k, hist_len):
    """the definition: GROUP BY kmer with collections.Counter, then GROUP BY count"""
    codes = O.np_generate(flat, off, k)
    per_kmer = collections.Counter(codes.tolist())
    hist = np.zeros(hist_len, np.uint64)
    tail = []
    for code, c in per_kmer.items():
        if c < hist_len:
            hist[c] += 1
        else:
            tail.append((code, c))
    tail.sort()
    return hist, np.array(tail, dtype=np.uint64).reshape(-1, 2)


@pytest.mark.parametrize("hist_len", [2, 3, 5, 64, 65536])
@pytest.mark.parametrize("k", [1, 3, 13, 21, 32])
def test_np_spectrum_equals_the_definition(k, hist_len):
    flat, off = datagen.synth_ragged(900 + k, 300, 120, min_len=32, mixed_case=True)
    rep = np.concatenate([flat, flat[:500], np.frombuffer(b"T" * 200 + b"A" * 90, np.uint8)])   # repeats, poly-T, poly-A
    roff = np.concatenate([off, [off[-1] + 500, off[-1] + 700, off[-1] + 790]]).astype(np.uint64)
    keys, counts, n = O.np_count(rep, roff, k)
    hist, tail = S.np_spectrum(keys, counts, hist_len)
    want_h, want_t = _counter_spectrum(rep, roff, k, hist_len)
    assert np.array_equal(hist, want_h) and np.array_equal(tail, want_t)
    # the invariant every GPU test asserts: sum c * hist[c] + sum of the tail's counts = windows
    assert int((np.arange(hist_len, dtype=np.uint64) * hist).sum()) + int(tail[:, 1].sum()) == n == rep.size - (roff.size - 1) * (k - 1)


def test_np_spectrum_equals_the_c_oracle_spectrum(corc):
    flat, off = datagen.synth_reads(77, 400, 150)
    flat = np.concatenate([flat, flat[:3000]])
    off = np.concatenate([off, off[1:21] + off[-1]]).astype(np.uint64)
    for k in (5, 14, 27):
        ck, cc, cn = corc.count(flat, off, k)
        keys, counts, n = O.np_count(flat, off, k)
        for hist_len in (2, 4, 1921):
            a = S.np_spectrum(ck, cc, hist_len)
            b = S.np_spectrum(keys, counts, hist_len)
            assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


@pytest.mark.parametrize("err", [0.0, 0.02])
@pytest.mark.parametrize("k", [21, 32])
def test_np_spectrum_of_the_coverage_oracle(k, err):
    """the spectrum of genome-sampled reads: the closed-form GROUP BY of coverage_util gives the same spectrum as a sort of every
    window; a poly-T run of 320 bases puts groups beyond a short histogram"""
    (flat, off), (genome, starts, err_pos) = CU.sample_reads(5000 + k + int(err * 100), 20_000, 1200, 300, err)
    lens = np.diff(off.astype(np.int64))
    keys, counts, n = CU.coverage_table(genome, starts, lens, err_pos, flat, k)
    ok, oc, on = O.np_count(flat, off, k)
    for hist_len in (2, 17, 65536):
        a, b = S.np_spectrum(keys, counts, hist_len), S.np_spectrum(ok, oc, hist_len)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    hist, tail = S.np_spectrum(keys, counts, 17)
    assert tail.shape[0] > 0 and hist[1] > 0 and hist[10:].sum() > 0    # coverage ~18: a real spectrum, and a tail


def test_spectrum_rows():
    z = np.zeros((0, 2), np.uint64)
    c, m = api.spectrum_rows(np.zeros(8, np.uint64), z)
    assert c.size == 0 and m.size == 0                                  # empty input: no rows
    c, m = api.spectrum_rows(np.zeros(2, np.uint64), np.array([[5, 9], [7, 2], [1, 9]], np.uint64))
    assert c.tolist() == [2, 9] and m.tolist() == [1, 2]                 # tail only; equal counts grouped
    hist = np.array([0, 10, 0, 4, 0, 0, 1], np.uint64)
    c, m = api.spectrum_rows(hist, np.array([[3, 7], [4, 100], [8, 7], [9, 7]], np.uint64))
    assert c.tolist() == [1, 3, 6, 7, 100] and m.tolist() == [10, 4, 1, 3, 1]   # zero bins omitted, ascending
    c, m = api.spectrum_rows(hist, np.array([7, 7, 100], np.uint64))    # a tail given as its counts
    assert c.tolist() == [1, 3, 6, 7, 100] and m.tolist() == [10, 4, 1, 2, 1]


@pytest.fixture(scope="module")
def lib():
    if not api.LIB_PATH.exists():
        import __graft_entry__ as g
        g.build()
    return api.load_library()


def test_spectrum_entry_points_reject_bad_arguments_without_touching_a_device(lib):
    """A NULL context, missing out-pointers or a histogram shorter than 2 come back as KMER_ERR_BAD_ARGUMENT before any CUDA
    call is made."""
    BAD = api.KMER_ERR_BAD_ARGUMENT
    vp = C.c_void_p
    hist, tail, nt, nk = vp(), vp(), C.c_uint64(), C.c_uint64()
    row = b"ACGTACGTACGTACGTACGTACGT"
    off = np.array([0, len(row)], np.uint64)
    for ctx in (None, vp(1)):       # a non-NULL context is never dereferenced on these paths
        assert lib.kmer_cuda_submit_count_spectrum(ctx, row, off.ctypes.data, 1, 21, 1, C.byref(hist), C.byref(tail), C.byref(nt),
                                                   C.byref(nk)) == BAD
        assert lib.kmer_cuda_submit_count_spectrum(ctx, row, off.ctypes.data, 1, 21, 16, None, C.byref(tail), C.byref(nt), None) == BAD
        assert lib.kmer_cuda_submit_count_spectrum(ctx, row, off.ctypes.data, 1, 21, 16, C.byref(hist), None, C.byref(nt), None) == BAD
        assert lib.kmer_cuda_submit_count_spectrum(ctx, row, off.ctypes.data, 1, 21, 16, C.byref(hist), C.byref(tail), None, None) == BAD
    assert lib.kmer_cuda_submit_count_spectrum(None, row, off.ctypes.data, 1, 21, 16, C.byref(hist), C.byref(tail), C.byref(nt),
                                               C.byref(nk)) == BAD
    assert lib.kmer_cuda_dev_count_spectrum(None, None, 0, None, 0, 21, None, 0, None, 0, 0, None) == BAD
    assert lib.kmer_cuda_dev_pairs_spectrum(None, None, 0, None, 0, None, 0, None) == BAD
    plan = api.KmerShardPlan()
    assert lib.kmer_cuda_dev_shard_count_spectrum(None, C.byref(plan), None, None, None, 0, None, 0, None) == BAD
    assert lib.kmer_cuda_dev_shard_count_spectrum(None, None, None, None, None, 16, None, 0, None) == BAD
