"""CPU checks of canonical counting's definition and oracles (tests/canonical_util.py), and of the new entry points' argument
checks (no device needed)."""
import ctypes as C

import numpy as np
import pytest

import canonical_util as CN
import coverage_util as CU
from kmer_extension_b200 import api
from oracle import oracle as O

RNG = np.random.default_rng(7)


def random_codes(k, n=2000):
    return RNG.integers(0, 1 << 63, n, dtype=np.uint64) * np.uint64(3) & np.uint64((1 << (2 * k)) - 1)


@pytest.mark.parametrize("k", range(1, 33))
def test_rc_is_an_involution_and_canon_is_the_smaller(k):
    x = random_codes(k)
    r = api.revcomp_codes(x, k)
    assert np.array_equal(api.revcomp_codes(r, k), x)
    c = api.canonical_codes(x, k)
    assert np.array_equal(c, api.canonical_codes(r, k)) and (c <= x).all() and (c <= r).all()
    if k < 32:
        assert (r < np.uint64(1 << (2 * k))).all()


@pytest.mark.parametrize("k", range(1, 33))
def test_code_rc_equals_text_rc(k):
    x = random_codes(k, 300)
    text = O.np_decode(x, k)
    want = [CN.rc_text(bytes(t).decode()) for t in text]
    got = [bytes(t).decode() for t in O.np_decode(api.revcomp_codes(x, k), k)]
    assert got == want
    assert [bytes(t).decode() for t in O.np_decode(api.canonical_codes(x, k), k)] == [CN.canon_text(bytes(t).decode()) for t in text]


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 6, 7, 8])
def test_palindromes_exist_only_at_even_k(k):
    x = np.arange(1 << (2 * k), dtype=np.uint64)
    pal = np.count_nonzero(api.revcomp_codes(x, k) == x)
    assert pal == (4 ** (k // 2) if k % 2 == 0 else 0)
    # every canonical class has one or two members: 4^k = 2 * classes - palindromes
    assert np.unique(api.canonical_codes(x, k)).size * 2 - pal == x.size


def test_k32_all_t_is_all_a():
    assert int(api.canonical_codes(np.array([~np.uint64(0)], np.uint64), 32)[0]) == 0
    assert int(api.canonical_codes(np.array([(1 << 52) - 1], np.uint64), 26)[0]) == 0    # t*26, the packed sentinel


def test_known_answers():
    for rows, k, want, spec in ((["ACGTACGT"], 4, {"acgt": 2, "cgta": 2, "gtac": 1}, {1: 1, 2: 2}),
                                (["ACGTT"], 3, {"aac": 1, "acg": 2}, None)):
        assert CN.text_count(rows, k) == want
        flat, off = O.rows_to_flat(rows)
        keys, counts, n = CN.np_canonical_count(flat, off, k)
        assert CN.counter_of(keys, counts, k) == want and n == sum(want.values())
        if spec:
            got = dict(zip(*np.unique(counts, return_counts=True)))
            assert {int(c): int(v) for c, v in got.items()} == spec


@pytest.mark.parametrize("k", [1, 2, 3, 5, 8, 13, 14, 15, 21, 26, 27, 31, 32])
def test_oracles_agree(corc, k):
    """text Counter == numpy codes == the C oracle's strand-specific count folded, on ragged mixed-case rows"""
    rng = np.random.default_rng(k)
    rows = []
    for i in range(60):
        n = int(rng.integers(k, k + 80))
        s = "".join("acgtACGT"[j] for j in rng.integers(0, 8, n))
        rows.append(s)
    rows += ["T" * (k + 9), "a" * (k + 3), "acgt" * (k // 4 + 3)]
    flat, off = O.rows_to_flat(rows)
    want = CN.text_count(rows, k)
    keys, counts, n = CN.np_canonical_count(flat, off, k)
    assert CN.counter_of(keys, counts, k) == want and n == sum(want.values())
    ck, cc, cn = corc.count(flat, off, k)
    ck_codes = O.np_encode_ascii(ck) if ck.ndim == 2 else ck
    fk, fc = CN.fold(ck_codes, cc, k)
    assert np.array_equal(fk, keys) and np.array_equal(fc, counts) and cn == n


@pytest.mark.parametrize("k,err,ragged", [(14, 0.0, False), (21, 0.002, True), (27, 0.02, False), (32, 0.002, True)])
def test_both_strand_closed_form(k, err, ragged):
    """reads from both strands with errors: the folded closed form equals the numpy canonical count, and poly-T / poly-A merge"""
    (flat, off), want = CN.both_strands(3, CU.MIN_GENOME * 2, 400, 150, k, err, ragged)
    got = CN.np_canonical_count(flat, off, k)
    assert got[2] == want[2] and np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    assert want[0][0] == 0                                       # a*k (and t*k, folded into it)


def test_revcomp_rows_is_an_involution_and_strand_invariant():
    rows = ["ACGTTGCAaacc", "gattacaGATTACA", "TTTTT"]
    flat, off = O.rows_to_flat(rows)
    f = np.frombuffer(flat, np.uint8) if isinstance(flat, (bytes, bytearray)) else flat
    which = np.array([True, False, True])
    r = CN.revcomp_rows(f, off, which)
    assert bytes(CN.revcomp_rows(r, off, which)) == bytes(f)
    assert bytes(r[:12]).decode() == "ggttTGCAACGT"
    for k in (2, 3, 5):
        a, b = CN.np_canonical_count(f, off, k), CN.np_canonical_count(r, off, k)
        assert all(np.array_equal(x, y) for x, y in zip(a[:2], b[:2]))


def test_new_entry_points_reject_bad_arguments():
    lib = api.load_library()
    vp, u = C.c_void_p, C.c_uint64
    hist, tail, n, nk = vp(), vp(), u(), u()
    assert lib.kmer_cuda_dev_count_canonical(None, None, 0, None, 0, 21, None, 0, None, 0, 0, None) == api.KMER_ERR_BAD_ARGUMENT
    assert lib.kmer_cuda_dev_count_canonical_spectrum(None, None, 0, None, 0, 21, None, 2, None, 0, 0, None) == api.KMER_ERR_BAD_ARGUMENT
    assert lib.kmer_cuda_submit_count_canonical(None, None, None, 0, 21, None, None, C.byref(tail), C.byref(n),
                                                C.byref(nk)) == api.KMER_ERR_BAD_ARGUMENT
    assert lib.kmer_cuda_submit_count_canonical_spectrum(None, None, None, 0, 21, 16, C.byref(hist), C.byref(tail), C.byref(n),
                                                         C.byref(nk)) == api.KMER_ERR_BAD_ARGUMENT
