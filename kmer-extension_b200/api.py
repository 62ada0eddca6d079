"""Host-side mirror of the reference's operator surface over libkmer_cuda.so (ctypes, no torch types
in any signature of the library; torch is used here only to own device buffers and streams).

The names and argument order follow the reference's SQL functions (kmer--1.0.0.sql:75-104):

    generate_kmers(dna, k)          -> codes of all windows            (generate_kmers, kmer.c:289-351)
    count_kmers(dna rows, k)        -> GROUP BY kmer / count(*)        (+ kmer_hash/kmer_equals, kmer.c:226-245,353-365)
    equals(kmer_col, kmer)          -> kmer = kmer                     (kmer_equals, kmer.c:226-245)
    starts_with(prefix, kmer_col)   -> starts_with(prefix, kmer)       (kmer_starts_with, kmer.c:248-255)
    starts_with_op(kmer_col, prefix)-> kmer ^@ prefix                  (kmer_starts_with_op, kmer.c:258-265)
    contains(qkmer, kmer_col)       -> qkmer @> kmer                   (kmer_contains, kmer.c:278-285)
    containing(kmer_col, qkmer)     -> kmer <@ qkmer                   (kmer_containing, kmer.c:268-275)

Errors surface as KmerSqlError carrying the reference's SQLSTATE, message and detail.
There is no CPU fallback: if libkmer_cuda.so is missing or no CUDA device is usable, constructing
the engine raises.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "libkmer_cuda.so"

KMER_OK = 0
KMER_ERR_INVALID_DNA, KMER_ERR_KMER_TOO_LONG, KMER_ERR_INVALID_QKMER, KMER_ERR_INVALID_K, KMER_ERR_QKMER_TOO_LONG = 1, 2, 3, 4, 5
KMER_ERR_BAD_ARGUMENT, KMER_ERR_CUDA, KMER_ERR_OOM, KMER_ERR_NO_DEVICE, KMER_ERR_CAPACITY = 16, 17, 18, 19, 20
OP_EQUALS, OP_STARTS_WITH, OP_CONTAINS = 0, 1, 2
ALGO_AUTO, ALGO_DENSE, ALGO_HASH, ALGO_PARTITION, ALGO_TWO_PASS = 0, 1, 2, 3, 4

# every symbol include/kmer_cuda.h declares (checked by tests/test_abi.py)
ABI_SYMBOLS = [
    "kmer_cuda_abi_version", "kmer_cuda_device_count", "kmer_cuda_init", "kmer_cuda_shutdown",
    "kmer_cuda_last_error", "kmer_cuda_release", "kmer_cuda_launch_count", "kmer_cuda_max_kmers",
    "kmer_cuda_submit_extract", "kmer_cuda_submit_count", "kmer_cuda_submit_match", "kmer_cuda_submit_decode",
    "kmer_cuda_submit_encode", "kmer_cuda_dev_extract", "kmer_cuda_dev_count", "kmer_cuda_dev_match",
    "kmer_cuda_dev_decode", "kmer_cuda_dev_finish", "kmer_cuda_set_profiling", "kmer_cuda_get_phases",
    "kmer_cuda_shard_plan", "kmer_cuda_dev_shard_partition", "kmer_cuda_dev_shard_count", "kmer_cuda_dev_dense_table",
    "kmer_cuda_dev_dense_emit", "kmer_cuda_submit_count_split", "kmer_cuda_dev_count_split", "kmer_cuda_submit_count_packed", "kmer_cuda_shard_plan_chunked", "kmer_cuda_dev_shard_count_split",
    "kmer_cuda_dev_shard_count_peers", "kmer_cuda_ipc_export", "kmer_cuda_ipc_open", "kmer_cuda_ipc_close",
    "kmer_cuda_dev_merge_begin", "kmer_cuda_dev_merge_add", "kmer_cuda_dev_merge_emit", "kmer_cuda_test_force_window",
    "kmer_cuda_init_multi", "kmer_cuda_shutdown_multi", "kmer_cuda_multi_device_count", "kmer_cuda_multi_last_error",
    "kmer_cuda_multi_submit_count", "kmer_cuda_multi_release", "kmer_cuda_dev_pack_codes", "kmer_cuda_multi_submit_match", "kmer_cuda_dev_synth_reads",
    "kmer_cuda_dev_count_spectrum", "kmer_cuda_dev_shard_count_spectrum", "kmer_cuda_dev_pairs_spectrum", "kmer_cuda_submit_count_spectrum",
    "kmer_cuda_dev_count_canonical", "kmer_cuda_dev_count_canonical_spectrum", "kmer_cuda_submit_count_canonical",
    "kmer_cuda_submit_count_canonical_spectrum",
]


class KmerCudaError(C.Structure):
    _fields_ = [("status", C.c_int), ("sqlstate", C.c_char * 6), ("message", C.c_char * 160),
                ("detail", C.c_char * 160), ("row", C.c_int64)]


class KmerDevResult(C.Structure):
    _fields_ = [("n_kmers", C.c_uint64), ("n_distinct", C.c_uint64), ("n_overflow", C.c_uint64), ("n_tier2", C.c_uint64),
                ("n_unique", C.c_uint64)]


class KmerShardPlan(C.Structure):
    _fields_ = [("n_ranks", C.c_uint32), ("n_buckets", C.c_uint32), ("buckets_per_rank", C.c_uint32), ("cap", C.c_uint32),
                ("k", C.c_int32), ("rec_bytes", C.c_int32), ("recs_bytes_per_peer", C.c_uint64),
                ("fill_bytes_per_peer", C.c_uint64), ("w", C.c_int32), ("m", C.c_int32), ("recw", C.c_int32), ("rmax", C.c_int32),
                ("fine_shift", C.c_uint32), ("fine_cap", C.c_uint32), ("chunks_per_rank", C.c_uint32), ("even_spread", C.c_uint32)]


class KmerSqlError(Exception):
    """An error of the engine, shaped like the reference's ereport(ERROR, ...)."""

    def __init__(self, status: int, sqlstate: str, message: str, detail: str, row: int):
        super().__init__(f"ERROR:  {message}" + (f"\nDETAIL:  {detail}" if detail else "") + f"  [{sqlstate}]")
        self.status, self.sqlstate, self.message, self.detail, self.row = status, sqlstate, message, detail, row


def load_library(path: Path = LIB_PATH) -> C.CDLL:
    if not Path(path).exists():
        raise FileNotFoundError(f"{path} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                                "(libkmer_cuda.so is the only compute path; there is no CPU fallback)")
    L = C.CDLL(str(path))
    u64, u64p, vp, i32, cp = C.c_uint64, C.POINTER(C.c_uint64), C.c_void_p, C.c_int, C.c_char_p
    L.kmer_cuda_abi_version.restype = i32
    L.kmer_cuda_device_count.restype = i32
    L.kmer_cuda_init.argtypes = [C.POINTER(vp), i32]
    L.kmer_cuda_shutdown.argtypes = [vp]
    L.kmer_cuda_shutdown.restype = None
    L.kmer_cuda_last_error.argtypes = [vp]
    L.kmer_cuda_last_error.restype = C.POINTER(KmerCudaError)
    L.kmer_cuda_release.argtypes = [vp, vp]
    L.kmer_cuda_release.restype = None
    L.kmer_cuda_launch_count.argtypes = [vp]
    L.kmer_cuda_launch_count.restype = u64
    L.kmer_cuda_max_kmers.argtypes = [u64, u64, i32]
    L.kmer_cuda_max_kmers.restype = u64
    L.kmer_cuda_submit_extract.argtypes = [vp, vp, vp, u64, i32, C.POINTER(vp), u64p]
    L.kmer_cuda_submit_count.argtypes = [vp, vp, vp, u64, i32, C.POINTER(vp), u64p, u64p]
    L.kmer_cuda_submit_match.argtypes = [vp, i32, vp, vp, vp, u64, i32, C.POINTER(cp), C.c_uint32, C.POINTER(vp), u64p, C.POINTER(vp)]
    L.kmer_cuda_submit_decode.argtypes = [vp, vp, u64, i32, i32, C.POINTER(vp)]
    L.kmer_cuda_submit_encode.argtypes = [vp, vp, vp, u64, i32, C.POINTER(vp)]
    L.kmer_cuda_dev_extract.argtypes = [vp, vp, u64, vp, u64, i32, vp, u64, vp]
    L.kmer_cuda_dev_count.argtypes = [vp, vp, u64, vp, u64, i32, vp, u64, i32, vp]
    L.kmer_cuda_dev_count_split.argtypes = [vp, vp, u64, vp, u64, i32, vp, u64, vp, u64, vp]
    L.kmer_cuda_submit_count_split.argtypes = [vp, vp, vp, u64, i32, C.POINTER(vp), u64p, C.POINTER(vp), u64p, u64p]
    L.kmer_cuda_submit_count_packed.argtypes = [vp, vp, vp, u64, i32, C.POINTER(vp), u64p, C.POINTER(C.c_int), C.POINTER(vp), u64p, u64p]
    L.kmer_cuda_dev_match.argtypes = [vp, i32, vp, vp, vp, u64, i32, C.POINTER(cp), C.c_uint32, vp, vp, vp]
    L.kmer_cuda_dev_decode.argtypes = [vp, vp, u64, i32, i32, vp, vp]
    L.kmer_cuda_dev_finish.argtypes = [vp, vp, C.POINTER(KmerDevResult)]
    L.kmer_cuda_set_profiling.argtypes = [vp, i32]
    L.kmer_cuda_set_profiling.restype = None
    L.kmer_cuda_get_phases.argtypes = [vp, C.POINTER(cp), C.POINTER(C.c_float), i32]
    L.kmer_cuda_shard_plan.argtypes = [u64, i32, C.c_uint32, C.POINTER(KmerShardPlan)]
    L.kmer_cuda_shard_plan_chunked.argtypes = [u64, i32, C.c_uint32, C.c_uint32, C.POINTER(KmerShardPlan)]
    L.kmer_cuda_dev_shard_partition.argtypes = [vp, vp, u64, vp, u64, C.POINTER(KmerShardPlan), vp, vp, vp]
    L.kmer_cuda_dev_shard_count.argtypes = [vp, C.POINTER(KmerShardPlan), vp, vp, vp, u64, vp]
    L.kmer_cuda_dev_shard_count_split.argtypes = [vp, C.POINTER(KmerShardPlan), vp, vp, vp, u64, vp, u64, vp]
    L.kmer_cuda_dev_shard_count_peers.argtypes = [vp, C.POINTER(KmerShardPlan), C.POINTER(vp), C.POINTER(vp), vp, u64, vp, u64, vp]
    L.kmer_cuda_ipc_export.argtypes = [vp, vp, C.c_char_p, C.POINTER(u64)]
    L.kmer_cuda_ipc_open.argtypes = [vp, C.c_char_p, C.POINTER(vp)]
    L.kmer_cuda_ipc_close.argtypes = [vp, vp]
    L.kmer_cuda_dev_dense_table.argtypes = [vp, vp, u64, vp, u64, i32, vp, vp]
    L.kmer_cuda_dev_dense_emit.argtypes = [vp, vp, i32, C.c_uint32, C.c_uint32, vp, u64, vp]
    L.kmer_cuda_test_force_window.argtypes = [i32]
    L.kmer_cuda_test_force_window.restype = None
    L.kmer_cuda_dev_pack_codes.argtypes = [vp, vp, u64, i32, vp, vp]
    L.kmer_cuda_dev_merge_begin.argtypes = [vp, u64, vp]
    L.kmer_cuda_dev_merge_add.argtypes = [vp, vp, u64, C.c_uint32, C.c_uint32, vp]
    L.kmer_cuda_dev_merge_emit.argtypes = [vp, i32, vp, u64, vp]
    L.kmer_cuda_dev_synth_reads.argtypes = [vp, u64, u64, u64, u64, vp, vp, vp]
    L.kmer_cuda_dev_count_spectrum.argtypes = [vp, vp, u64, vp, u64, i32, vp, u64, vp, u64, i32, vp]
    L.kmer_cuda_dev_shard_count_spectrum.argtypes = [vp, C.POINTER(KmerShardPlan), C.POINTER(vp), C.POINTER(vp), vp, u64, vp, u64, vp]
    L.kmer_cuda_dev_pairs_spectrum.argtypes = [vp, vp, u64, vp, u64, vp, u64, vp]
    L.kmer_cuda_submit_count_spectrum.argtypes = [vp, vp, vp, u64, i32, u64, C.POINTER(vp), C.POINTER(vp), u64p, u64p]
    L.kmer_cuda_dev_count_canonical.argtypes = [vp, vp, u64, vp, u64, i32, vp, u64, vp, u64, i32, vp]
    L.kmer_cuda_dev_count_canonical_spectrum.argtypes = [vp, vp, u64, vp, u64, i32, vp, u64, vp, u64, i32, vp]
    L.kmer_cuda_submit_count_canonical.argtypes = [vp, vp, vp, u64, i32, C.POINTER(vp), u64p, C.POINTER(vp), u64p, u64p]
    L.kmer_cuda_submit_count_canonical_spectrum.argtypes = [vp, vp, vp, u64, i32, u64, C.POINTER(vp), C.POINTER(vp), u64p, u64p]
    return L


def _flat(rows_or_flat, off=None):
    """Accept (flat uint8 array/bytes, offsets) or a list of str/bytes rows."""
    if off is not None:
        f = np.frombuffer(rows_or_flat, dtype=np.uint8) if isinstance(rows_or_flat, (bytes, bytearray)) else \
            np.ascontiguousarray(rows_or_flat, dtype=np.uint8)
        return f, np.ascontiguousarray(off, dtype=np.uint64)
    bs = [r.encode() if isinstance(r, str) else bytes(r) for r in rows_or_flat]
    o = np.zeros(len(bs) + 1, dtype=np.uint64)
    if bs:
        o[1:] = np.cumsum([len(b) for b in bs], dtype=np.uint64)
    return np.frombuffer(b"".join(bs), dtype=np.uint8), o


def revcomp_codes(codes, k: int) -> np.ndarray:
    """Codes of the reverse complements (a<->t, c<->g, order reversed) of k-mer codes (numpy, uint64)."""
    x = ~np.asarray(codes, dtype=np.uint64)
    r = np.zeros_like(x)
    for i in range(k):                                          # base i (from the first) becomes base k-1-i
        r |= ((x >> np.uint64(2 * (k - 1 - i))) & np.uint64(3)) << np.uint64(2 * i)
    return r


def canonical_codes(codes, k: int) -> np.ndarray:
    """min(code, reverse complement): the group key of canonical counting."""
    c = np.asarray(codes, dtype=np.uint64)
    return np.minimum(c, revcomp_codes(c, k))


def spectrum_rows(hist, tail):
    """The SQL relation of the abundance spectrum -- `SELECT cnt AS count, count(*) AS kmers FROM (... GROUP BY kmer) s GROUP BY
    cnt ORDER BY cnt` -- from a histogram (hist[c] = k-mers counted c times, c < len(hist)) and the tail of groups whose count is
    >= len(hist) (an [n, 2] (code, count) array, or just their counts): (count, kmers) uint64 arrays, ascending by count, zero
    rows omitted."""
    hist = np.asarray(hist, dtype=np.uint64).reshape(-1)
    tail = np.asarray(tail, dtype=np.uint64)
    tcounts = tail[:, 1] if tail.ndim == 2 else tail.reshape(-1)
    c = np.nonzero(hist)[0].astype(np.uint64)
    tc, tk = np.unique(tcounts, return_counts=True)
    return np.concatenate([c, tc.astype(np.uint64)]), np.concatenate([hist[c.astype(np.int64)], tk.astype(np.uint64)])


class KmerCuda:
    """One engine context on one GPU (process-local, one batch in flight)."""

    def __init__(self, device: int = 0, lib_path: Path = LIB_PATH):
        self.lib = load_library(lib_path)
        self.ctx = C.c_void_p()
        rc = self.lib.kmer_cuda_init(C.byref(self.ctx), device)
        if rc:
            self._raise(None)
        self.device = device

    # ------------------------------------------------------------------ plumbing
    def close(self):
        if getattr(self, "ctx", None) and self.ctx.value:
            self.lib.kmer_cuda_shutdown(self.ctx)
            self.ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _raise(self, ctx):
        e = self.lib.kmer_cuda_last_error(ctx).contents
        raise KmerSqlError(e.status, e.sqlstate.decode(), e.message.decode(), e.detail.decode(), e.row)

    def _check(self, rc):
        if rc:
            self._raise(self.ctx)

    @property
    def launches(self) -> int:
        return int(self.lib.kmer_cuda_launch_count(self.ctx))

    def set_profiling(self, on: bool):
        self.profiling = bool(on)
        self.lib.kmer_cuda_set_profiling(self.ctx, int(on))

    def phases(self) -> list[tuple[str, float]]:
        """(phase name, device ms) of the last finished dev_* call (needs set_profiling(True))."""
        names = (C.c_char_p * 64)()
        ms = (C.c_float * 64)()
        n = self.lib.kmer_cuda_get_phases(self.ctx, names, ms, 64)
        return [(names[i].decode(), float(ms[i])) for i in range(min(n, 64))]

    def max_kmers(self, n_bases: int, n_rows: int, k: int) -> int:
        return int(self.lib.kmer_cuda_max_kmers(n_bases, n_rows, k))

    def _take(self, ptr: C.c_void_p, nbytes: int, dtype, copy=True) -> np.ndarray:
        """View a library-owned pinned result as numpy, copy it out and release it."""
        if nbytes == 0 or not ptr.value:
            if ptr.value:
                self.lib.kmer_cuda_release(self.ctx, ptr)
            return np.zeros(0, dtype=dtype)
        buf = (C.c_char * nbytes).from_address(ptr.value)
        a = np.frombuffer(buf, dtype=dtype)
        if copy:
            a = a.copy()
            self.lib.kmer_cuda_release(self.ctx, ptr)
        return a

    # ------------------------------------------------------------------ host-buffer batch submit
    def generate_kmers(self, rows_or_flat, k: int, off=None) -> np.ndarray:
        """All windows of all rows, rows in order, positions in order -> uint64 codes."""
        f, o = _flat(rows_or_flat, off)
        codes, n = C.c_void_p(), C.c_uint64()
        self._check(self.lib.kmer_cuda_submit_extract(self.ctx, f.ctypes.data, o.ctypes.data, len(o) - 1, k,
                                                      C.byref(codes), C.byref(n)))
        return self._take(codes, n.value * 8, np.uint64)

    def count_kmers(self, rows_or_flat, k: int, off=None, canonical: bool = False):
        """GROUP BY kmer / count(*) -> (codes[D] uint64, counts[D] uint64, n_kmers); order unspecified.  canonical: a k-mer and
        its reverse complement are one group, keyed by canonical_codes()."""
        f, o = _flat(rows_or_flat, off)
        pairs, d, n = C.c_void_p(), C.c_uint64(), C.c_uint64()
        if canonical:
            self._check(self.lib.kmer_cuda_submit_count_canonical(self.ctx, f.ctypes.data, o.ctypes.data, len(o) - 1, k, None, None,
                                                                  C.byref(pairs), C.byref(d), C.byref(n)))
        else:
            self._check(self.lib.kmer_cuda_submit_count(self.ctx, f.ctypes.data, o.ctypes.data, len(o) - 1, k,
                                                        C.byref(pairs), C.byref(d), C.byref(n)))
        a = self._take(pairs, d.value * 16, np.uint64).reshape(-1, 2)
        return a[:, 0].copy(), a[:, 1].copy(), int(n.value)

    def count_kmers_split(self, rows_or_flat, k: int, off=None, canonical: bool = False):
        """The same GROUP BY in the split format -> (unique codes[U], codes[P], counts[P], n_kmers)."""
        f, o = _flat(rows_or_flat, off)
        uq, nu, pairs, npairs, n = C.c_void_p(), C.c_uint64(), C.c_void_p(), C.c_uint64(), C.c_uint64()
        fn = self.lib.kmer_cuda_submit_count_canonical if canonical else self.lib.kmer_cuda_submit_count_split
        self._check(fn(self.ctx, f.ctypes.data, o.ctypes.data, len(o) - 1, k, C.byref(uq), C.byref(nu), C.byref(pairs),
                       C.byref(npairs), C.byref(n)))
        u = self._take(uq, nu.value * 8, np.uint64)
        a = self._take(pairs, npairs.value * 16, np.uint64).reshape(-1, 2)
        return u.copy(), a[:, 0].copy(), a[:, 1].copy(), int(n.value)

    def count_kmers_packed(self, rows_or_flat, k: int, off=None):
        """Split format with packed bare codes -> (unique codes[U] (unpacked here), codes[P], counts[P], n_kmers, code_bytes)."""
        f, o = _flat(rows_or_flat, off)
        uq, nu, nb, pairs, npairs, n = C.c_void_p(), C.c_uint64(), C.c_int(), C.c_void_p(), C.c_uint64(), C.c_uint64()
        self._check(self.lib.kmer_cuda_submit_count_packed(self.ctx, f.ctypes.data, o.ctypes.data, len(o) - 1, k, C.byref(uq),
                                                           C.byref(nu), C.byref(nb), C.byref(pairs), C.byref(npairs), C.byref(n)))
        raw = self._take(uq, nu.value * nb.value, np.uint8).reshape(-1, max(nb.value, 1))
        u = np.zeros(raw.shape[0], dtype=np.uint64)
        for b in range(nb.value):
            u |= raw[:, b].astype(np.uint64) << np.uint64(8 * b)
        a = self._take(pairs, npairs.value * 16, np.uint64).reshape(-1, 2)
        return u, a[:, 0].copy(), a[:, 1].copy(), int(n.value), int(nb.value)

    def count_spectrum(self, rows_or_flat, k: int, off=None, hist_len: int = 65536, canonical: bool = False):
        """Abundance spectrum of the GROUP BY -> (hist[hist_len] uint64, tail [n, 2] uint64 (code, count) of the groups with
        count >= hist_len, order unspecified); spectrum_rows(hist, tail) is the SQL relation."""
        f, o = _flat(rows_or_flat, off)
        hist, tail, nt, n = C.c_void_p(), C.c_void_p(), C.c_uint64(), C.c_uint64()
        fn = self.lib.kmer_cuda_submit_count_canonical_spectrum if canonical else self.lib.kmer_cuda_submit_count_spectrum
        self._check(fn(self.ctx, f.ctypes.data, o.ctypes.data, len(o) - 1, k, hist_len, C.byref(hist), C.byref(tail), C.byref(nt),
                       C.byref(n)))
        h = self._take(hist, hist_len * 8, np.uint64)
        t = self._take(tail, nt.value * 16, np.uint64).reshape(-1, 2)
        return h, t

    def match(self, op, codes: np.ndarray, k: int, consts, lens: np.ndarray | None = None, ops=None):
        """Bit matrix [n_consts, m] (bool) and hits[n_consts] for the column `codes`."""
        codes = np.ascontiguousarray(codes, dtype=np.uint64)
        m = codes.size
        consts = [consts] if isinstance(consts, str) else list(consts)
        arr = (C.c_char_p * max(len(consts), 1))(*[s.encode() for s in consts])
        lp = None
        if lens is not None:
            lens = np.ascontiguousarray(lens, dtype=np.uint8)
            lp = lens.ctypes.data
        opsp = None
        if ops is not None:
            ops_a = np.ascontiguousarray(ops, dtype=np.int32)
            opsp = ops_a.ctypes.data
        bits, wpr, hits = C.c_void_p(), C.c_uint64(), C.c_void_p()
        self._check(self.lib.kmer_cuda_submit_match(self.ctx, op, opsp, codes.ctypes.data, lp, m, k, arr, len(consts),
                                                    C.byref(bits), C.byref(wpr), C.byref(hits)))
        w = self._take(bits, len(consts) * wpr.value * 4, np.uint32).reshape(len(consts), wpr.value)
        h = self._take(hits, len(consts) * 8, np.uint64)
        if m == 0:
            return np.zeros((len(consts), 0), dtype=bool), h
        unpacked = np.unpackbits(w.view(np.uint8), axis=1, bitorder="little")[:, :m].astype(bool)
        return unpacked, h

    # SQL-named forms (single constant) ------------------------------------------------------------
    def equals(self, kmer_col, kmer: str, k: int, lens=None) -> np.ndarray:
        return self.match(OP_EQUALS, kmer_col, k, kmer, lens)[0][0]

    def starts_with(self, prefix: str, kmer_col, k: int, lens=None) -> np.ndarray:
        return self.match(OP_STARTS_WITH, kmer_col, k, prefix, lens)[0][0]

    def starts_with_op(self, kmer_col, prefix: str, k: int, lens=None) -> np.ndarray:
        return self.match(OP_STARTS_WITH, kmer_col, k, prefix, lens)[0][0]

    def contains(self, qkmer: str, kmer_col, k: int, lens=None) -> np.ndarray:
        return self.match(OP_CONTAINS, kmer_col, k, qkmer, lens)[0][0]

    def containing(self, kmer_col, qkmer: str, k: int, lens=None) -> np.ndarray:
        return self.match(OP_CONTAINS, kmer_col, k, qkmer, lens)[0][0]

    def decode(self, codes: np.ndarray, k: int, with_header: bool = False) -> np.ndarray:
        """codes -> [n, k(+1)] uint8 text as the reference stores it (kmer_out / short varlena header)."""
        codes = np.ascontiguousarray(codes, dtype=np.uint64)
        text = C.c_void_p()
        self._check(self.lib.kmer_cuda_submit_decode(self.ctx, codes.ctypes.data, codes.size, k, int(with_header), C.byref(text)))
        rec = k + (1 if with_header else 0)
        return self._take(text, codes.size * rec, np.uint8).reshape(codes.size, rec) if rec else np.zeros((codes.size, 0), np.uint8)

    def encode(self, text: np.ndarray, lens: np.ndarray | None = None) -> np.ndarray:
        """[n, stride] uint8 k-mer text -> codes (batched kmer_in)."""
        text = np.ascontiguousarray(text, dtype=np.uint8)
        n, stride = text.shape
        lp = None
        if lens is not None:
            lens = np.ascontiguousarray(lens, dtype=np.uint8)
            lp = lens.ctypes.data
        codes = C.c_void_p()
        self._check(self.lib.kmer_cuda_submit_encode(self.ctx, text.ctypes.data, lp, n, stride, C.byref(codes)))
        return self._take(codes, n * 8, np.uint64)

    # ------------------------------------------------------------------ device-resident API (torch owns the buffers)
    @staticmethod
    def _stream_ptr(stream=None):
        import torch
        s = stream if stream is not None else torch.cuda.current_stream()
        return C.c_void_p(s.cuda_stream)

    def dev_extract(self, d_seq, n_bases: int, d_off, n_rows: int, k: int, d_codes, stream=None):
        self._check(self.lib.kmer_cuda_dev_extract(self.ctx, d_seq.data_ptr(), n_bases, d_off.data_ptr(), n_rows, k,
                                                   d_codes.data_ptr(), d_codes.numel(), self._stream_ptr(stream)))

    def dev_count(self, d_seq, n_bases: int, d_off, n_rows: int, k: int, d_pairs, algo: int = ALGO_AUTO, stream=None,
                  canonical: bool = False):
        """d_pairs: int64/uint64 tensor [capacity, 2].  canonical: canonical k-mers (ALGO_TWO_PASS runs as ALGO_PARTITION)."""
        if canonical:
            self._check(self.lib.kmer_cuda_dev_count_canonical(self.ctx, d_seq.data_ptr(), n_bases, d_off.data_ptr(), n_rows, k, None, 0,
                                                               d_pairs.data_ptr(), d_pairs.numel() // 2, algo, self._stream_ptr(stream)))
            return
        self._check(self.lib.kmer_cuda_dev_count(self.ctx, d_seq.data_ptr(), n_bases, d_off.data_ptr(), n_rows, k,
                                                 d_pairs.data_ptr(), d_pairs.numel() // 2, algo, self._stream_ptr(stream)))

    def dev_count_split(self, d_seq, n_bases: int, d_off, n_rows: int, k: int, d_uniq, d_pairs, stream=None, canonical: bool = False):
        """d_uniq: uint64/int64 tensor [capacity]; d_pairs: [capacity, 2]."""
        if canonical:
            self._check(self.lib.kmer_cuda_dev_count_canonical(self.ctx, d_seq.data_ptr(), n_bases, d_off.data_ptr(), n_rows, k,
                                                               d_uniq.data_ptr(), d_uniq.numel(), d_pairs.data_ptr(), d_pairs.numel() // 2,
                                                               ALGO_AUTO, self._stream_ptr(stream)))
            return
        self._check(self.lib.kmer_cuda_dev_count_split(self.ctx, d_seq.data_ptr(), n_bases, d_off.data_ptr(), n_rows, k,
                                                       d_uniq.data_ptr(), d_uniq.numel(), d_pairs.data_ptr(), d_pairs.numel() // 2,
                                                       self._stream_ptr(stream)))

    def dev_count_spectrum(self, d_seq, n_bases: int, d_off, n_rows: int, k: int, d_hist, d_tail, algo: int = ALGO_AUTO, stream=None,
                           canonical: bool = False):
        """Spectrum result format: d_hist uint64/int64 [hist_len] (overwritten whole), d_tail [tail_capacity, 2] gets the groups
        with count >= hist_len; dev_finish().n_distinct = tail entries written."""
        fn = self.lib.kmer_cuda_dev_count_canonical_spectrum if canonical else self.lib.kmer_cuda_dev_count_spectrum
        self._check(fn(self.ctx, d_seq.data_ptr(), n_bases, d_off.data_ptr(), n_rows, k, d_hist.data_ptr(), d_hist.numel(),
                       d_tail.data_ptr(), d_tail.shape[0], algo, self._stream_ptr(stream)))

    def dev_pairs_spectrum(self, d_pairs, n: int, d_hist, d_tail, stream=None):
        """The spectrum of the (code, count) table d_pairs[:n] (same outputs as dev_count_spectrum)."""
        self._check(self.lib.kmer_cuda_dev_pairs_spectrum(self.ctx, d_pairs.data_ptr(), n, d_hist.data_ptr(), d_hist.numel(),
                                                          d_tail.data_ptr(), d_tail.shape[0], self._stream_ptr(stream)))

    def dev_match(self, op, d_codes, m: int, k: int, consts, d_bits, d_hits, d_lens=None, ops=None, stream=None):
        consts = [consts] if isinstance(consts, str) else list(consts)
        arr = (C.c_char_p * max(len(consts), 1))(*[s.encode() for s in consts])
        opsp = None
        if ops is not None:
            ops_a = np.ascontiguousarray(ops, dtype=np.int32)
            opsp = ops_a.ctypes.data
        self._check(self.lib.kmer_cuda_dev_match(self.ctx, op, opsp, d_codes.data_ptr(),
                                                 d_lens.data_ptr() if d_lens is not None else None, m, k, arr, len(consts),
                                                 d_bits.data_ptr(), d_hits.data_ptr(), self._stream_ptr(stream)))

    def dev_synth_reads(self, seed: int, first_row: int, n_rows: int, read_len: int, d_seq, d_off, stream=None):
        """Rows [first_row, first_row+n_rows) of the seeded synthetic table, written into d_seq (uint8, >= n_rows*read_len
        rounded up to 16 bytes) and d_off (int64/uint64 [n_rows+1]); datagen.synth_reads_counter is the numpy restatement."""
        self._check(self.lib.kmer_cuda_dev_synth_reads(self.ctx, seed & ((1 << 64) - 1), first_row, n_rows, read_len, d_seq.data_ptr(),
                                                       d_off.data_ptr(), self._stream_ptr(stream)))

    def dev_decode(self, d_codes, n: int, k: int, with_header: bool, d_text, stream=None):
        self._check(self.lib.kmer_cuda_dev_decode(self.ctx, d_codes.data_ptr(), n, k, int(with_header), d_text.data_ptr(),
                                                  self._stream_ptr(stream)))

    # ------------------------------------------------------------------ sharded counting (the caller runs the exchange)
    def shard_plan(self, total_kmers: int, k: int, n_ranks: int, chunks: int = 1) -> KmerShardPlan:
        plan = KmerShardPlan()
        if self.lib.kmer_cuda_shard_plan_chunked(total_kmers, k, n_ranks, chunks, C.byref(plan)):
            raise ValueError("kmer_cuda_shard_plan: needs 14 <= k <= 32 and n_ranks >= 1")
        return plan

    def dev_shard_partition(self, d_seq, n_bases: int, d_off, n_rows: int, plan: KmerShardPlan, d_send_recs, d_send_fill, stream=None):
        self._check(self.lib.kmer_cuda_dev_shard_partition(self.ctx, d_seq.data_ptr(), n_bases, d_off.data_ptr(), n_rows,
                                                           C.byref(plan), d_send_recs.data_ptr(), d_send_fill.data_ptr(),
                                                           self._stream_ptr(stream)))

    def dev_shard_count(self, plan: KmerShardPlan, d_recv_recs, d_recv_fill, d_pairs, stream=None):
        self._check(self.lib.kmer_cuda_dev_shard_count(self.ctx, C.byref(plan), d_recv_recs.data_ptr(), d_recv_fill.data_ptr(),
                                                       d_pairs.data_ptr(), d_pairs.numel() // 2, self._stream_ptr(stream)))

    def dev_shard_count_split(self, plan: KmerShardPlan, d_recv_recs, d_recv_fill, d_uniq, d_pairs, stream=None):
        self._check(self.lib.kmer_cuda_dev_shard_count_split(self.ctx, C.byref(plan), d_recv_recs.data_ptr(), d_recv_fill.data_ptr(),
                                                             d_uniq.data_ptr(), d_uniq.numel(), d_pairs.data_ptr(), d_pairs.numel() // 2,
                                                             self._stream_ptr(stream)))

    def dev_shard_count_peers(self, plan: KmerShardPlan, src_recs, src_fill, d_uniq, d_pairs, stream=None):
        """src_recs / src_fill: device ADDRESSES (ints) of every source's segments for this rank (kmer_cuda.h)."""
        n = len(src_recs)
        a_r = (C.c_void_p * n)(*[int(x) for x in src_recs])
        a_f = (C.c_void_p * n)(*[int(x) for x in src_fill])
        self._check(self.lib.kmer_cuda_dev_shard_count_peers(
            self.ctx, C.byref(plan), a_r, a_f, d_uniq.data_ptr() if d_uniq is not None else None,
            d_uniq.numel() if d_uniq is not None else 0, d_pairs.data_ptr(), d_pairs.numel() // 2, self._stream_ptr(stream)))

    def dev_shard_count_spectrum(self, plan: KmerShardPlan, src_recs, src_fill, d_hist, d_tail, stream=None):
        """This rank's share in the spectrum format; src_recs / src_fill: device ADDRESSES (ints) of every source's segments for
        this rank -- the peers' send blocks, or recv_recs + s * recs_bytes_per_peer / recv_fill + s * buckets_per_rank * 8."""
        n = len(src_recs)
        a_r = (C.c_void_p * n)(*[int(x) for x in src_recs])
        a_f = (C.c_void_p * n)(*[int(x) for x in src_fill])
        self._check(self.lib.kmer_cuda_dev_shard_count_spectrum(self.ctx, C.byref(plan), a_r, a_f, d_hist.data_ptr(), d_hist.numel(),
                                                                d_tail.data_ptr(), d_tail.shape[0], self._stream_ptr(stream)))

    def ipc_export(self, d_tensor):
        """(64-byte handle of the allocation the tensor lies in, the tensor's byte offset inside it)"""
        h = C.create_string_buffer(64)
        off = C.c_uint64(0)
        self._check(self.lib.kmer_cuda_ipc_export(self.ctx, d_tensor.data_ptr(), h, C.byref(off)))
        return bytes(h.raw), int(off.value)

    def ipc_open(self, handle: bytes) -> int:
        base = C.c_void_p(0)
        self._check(self.lib.kmer_cuda_ipc_open(self.ctx, handle, C.byref(base)))
        return int(base.value)

    def ipc_close(self, base: int):
        self._check(self.lib.kmer_cuda_ipc_close(self.ctx, base))

    def dev_pack_codes(self, d_codes, n: int, k: int, d_packed, stream=None):
        self._check(self.lib.kmer_cuda_dev_pack_codes(self.ctx, d_codes.data_ptr(), n, k, d_packed.data_ptr(), self._stream_ptr(stream)))

    def dev_merge_begin(self, max_groups: int, stream=None):
        self._check(self.lib.kmer_cuda_dev_merge_begin(self.ctx, max_groups, self._stream_ptr(stream)))

    def dev_merge_add(self, d_pairs, n: int, rank: int, n_ranks: int, stream=None):
        self._check(self.lib.kmer_cuda_dev_merge_add(self.ctx, d_pairs.data_ptr(), n, rank, n_ranks, self._stream_ptr(stream)))

    def dev_merge_emit(self, k: int, d_pairs, stream=None):
        self._check(self.lib.kmer_cuda_dev_merge_emit(self.ctx, k, d_pairs.data_ptr(), d_pairs.numel() // 2, self._stream_ptr(stream)))

    def dev_dense_table(self, d_seq, n_bases: int, d_off, n_rows: int, k: int, d_table, stream=None):
        self._check(self.lib.kmer_cuda_dev_dense_table(self.ctx, d_seq.data_ptr(), n_bases, d_off.data_ptr(), n_rows, k,
                                                       d_table.data_ptr(), self._stream_ptr(stream)))

    def dev_dense_emit(self, d_table, k: int, rank: int, n_ranks: int, d_pairs, stream=None):
        self._check(self.lib.kmer_cuda_dev_dense_emit(self.ctx, d_table.data_ptr(), k, rank, n_ranks, d_pairs.data_ptr(),
                                                      d_pairs.numel() // 2, self._stream_ptr(stream)))

    def dev_finish(self, stream=None) -> KmerDevResult:
        r = KmerDevResult()
        self._check(self.lib.kmer_cuda_dev_finish(self.ctx, self._stream_ptr(stream), C.byref(r)))
        return r
