"""Helpers shared by the parity tests: load fixtures, regenerate their seeded inputs, canonical hashes."""
import hashlib
import json
from pathlib import Path

import numpy as np

import conftest  # noqa: F401  (loads the hyphenated package)
from kmer_extension_b200 import datagen
from oracle import oracle as O

GOLDEN = Path(__file__).resolve().parent / "golden"


def load(name):
    return json.loads((GOLDEN / name).read_text())


def sha(b: bytes) -> str:
    return hashlib.sha256(b).hexdigest()


def make_input(spec):
    if spec["gen"] == "reads":
        return datagen.synth_reads(spec["seed"], spec["n_rows"], spec["read_len"])
    return datagen.synth_ragged(spec["seed"], spec["n_rows"], spec["max_len"], spec.get("min_len", 1),
                                mixed_case=spec.get("mixed_case", False))


def checked_input(case):
    flat, off = make_input(case["input"])
    assert sha(flat.tobytes()) == case["input_sha256"], "datagen no longer reproduces the fixture's input bytes"
    return flat, off


def count_canon_from_codes(keys: np.ndarray, counts: np.ndarray, k: int) -> bytes:
    """canonical serialisation of a (code,count) table: b'<kmer>:<count>\\n' sorted by k-mer text."""
    keys = np.asarray(keys, dtype=np.uint64)
    counts = np.asarray(counts, dtype=np.uint64)
    order = np.argsort(keys, kind="stable")  # code order == text order for equal k
    txt = O.np_decode(keys[order], k)
    cs = counts[order]
    return b"".join(bytes(t) + b":" + str(int(c)).encode() + b"\n" for t, c in zip(txt, cs))


def generate_canon_from_codes(codes: np.ndarray, k: int) -> bytes:
    return O.np_decode(codes, k).tobytes()


def expected_side_link_args() -> list:
    """gcc arguments for the expected side of tests/c/{glue,hook}_driver.c (tests/c/expected_kmers.h): the reference's own
    functions where oracle/_ref is built, else the C oracle (pinned to the reference's answers by test_oracle.py) with the
    pgshim runtime of oracle/ref_driver.c"""
    O.build(ref=True)
    if O.REF_SO.exists():
        return [f"-L{O.REF_SO.parent}", "-lkmer_ref", f"-Wl,-rpath,{O.REF_SO.parent}"]
    return ["-DPGSHIM_NO_REFERENCE", "-Wno-unused-function", str(O.HERE / "ref_driver.c"), f"-L{O.HERE}", "-lkmer_oracle",
            f"-Wl,-rpath,{O.HERE}"]
