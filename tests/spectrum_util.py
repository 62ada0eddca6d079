"""The abundance spectrum (count of counts) of a GROUP BY table, restated in numpy: what the spectrum entry points of
libkmer_cuda.so must return for the same rows (include/kmer_cuda.h, kmer_cuda_dev_count_spectrum)."""
import numpy as np


def np_spectrum(keys, counts, hist_len):
    """(keys, counts) of `SELECT kmer, count(*) ... GROUP BY kmer` -> (hist[hist_len] uint64, tail [n, 2] uint64 sorted by code):
    hist[c] = number of k-mers counted exactly c times for c < hist_len (hist[0] = 0), tail = the groups with count >= hist_len."""
    keys = np.asarray(keys, dtype=np.uint64)
    counts = np.asarray(counts, dtype=np.uint64)
    small = counts < np.uint64(hist_len)
    hist = np.bincount(counts[small].astype(np.int64), minlength=hist_len).astype(np.uint64)[:hist_len]
    hist[0] = 0
    tk, tc = keys[~small], counts[~small]
    o = np.argsort(tk, kind="stable")
    return hist, np.stack([tk[o], tc[o]], axis=1) if tk.size else np.zeros((0, 2), np.uint64)


def sorted_tail(tail):
    """a tail in unspecified order (uint64 or int64 [n, 2]) -> uint64 [n, 2] sorted by code"""
    t = np.ascontiguousarray(tail).reshape(-1, 2)
    t = t.view(np.uint64) if t.dtype == np.int64 else t.astype(np.uint64)
    return t[np.argsort(t[:, 0], kind="stable")]
