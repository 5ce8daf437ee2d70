"""Records what the reference tree's own code computes on the inputs of three tests, so that those tests compare with it
wherever they run:
  edlib_hw_distance.npz  edlib's infix edit distance for every case of tests/test_dp_vs_edlib.py
  kseq_records.json      kseq++'s records (count, block digests) for every file of tests/test_reader_vs_kseq.py
  eigen_digamma.npz      Eigen's digamma at a seeded sample of the arguments tests/test_math_pinning.py used to draw
It loads the libraries oracle/build_ref.sh compiles into oracle/_ref/ from a reference source tree, and it runs the edlib
and kseq++ tests while it records, so the product must be built.
Run: python tests/golden/make_ref_golden.py"""
import ctypes as C
import json
import os
import sys
import tempfile
from pathlib import Path

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.path.join(ROOT, "oracle", "_ref")
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import test_dp_vs_edlib as E      # noqa: E402
import test_reader_vs_kseq as K   # noqa: E402


class EdlibAlignConfig(C.Structure):
    _fields_ = [("k", C.c_int), ("mode", C.c_int), ("task", C.c_int)]


class EdlibAlignResult(C.Structure):
    _fields_ = [("editDistance", C.c_int), ("endLocations", C.POINTER(C.c_int)), ("startLocations", C.POINTER(C.c_int)),
                ("numLocations", C.c_int), ("alignment", C.POINTER(C.c_ubyte)), ("alignmentLength", C.c_int),
                ("alphabetLength", C.c_int)]


def record_edlib():
    lib = C.CDLL(os.path.join(REF, "libedlib_ref.so"))
    align = getattr(lib, "_Z10edlibAlignPKciS0_i16EdlibAlignConfig")      # edlibAlign(const char*, int, const char*, int, EdlibAlignConfig)
    align.restype = EdlibAlignResult
    align.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, EdlibAlignConfig]
    free = getattr(lib, "_Z20edlibFreeAlignResult16EdlibAlignResult")
    free.restype = None
    free.argtypes = [EdlibAlignResult]
    seen = {}

    def hw_distance(query: bytes, target: bytes) -> int:
        r = align(query, len(query), target, len(target), EdlibAlignConfig(-1, 2, 0))     # k = -1, EDLIB_MODE_HW, TASK_DISTANCE
        d = r.editDistance
        free(r)
        seen[E.hw_key(query, target)] = d
        return d
    E._edlib = lambda: hw_distance
    for test in (E.test_unit_cost_dp_equals_edlib_infix_distance, E.test_default_scores_bound_by_edit_distance,
                 E.test_product_serial_dp_equals_edlib_and_oracle):
        test()
    np.savez(E.GOLDEN, key=np.array(list(seen), np.uint64), dist=np.array(list(seen.values()), np.int32))
    print(E.GOLDEN, len(seen), "cases")


def record_kseq():
    lib = C.CDLL(os.path.join(REF, "libkseq_ref.so"))
    lib.ref_kseq_parse.restype = C.c_long
    seen = {}

    def kseq(path):
        tot = C.c_ulong(0)
        n = lib.ref_kseq_parse(os.fsencode(path), None, C.c_ulong(0), None, C.c_ulong(0), C.byref(tot))
        assert n >= 0
        seq = np.empty(max(tot.value, 1), np.uint8)
        lens = np.empty(max(n, 1), np.uint32)
        n2 = lib.ref_kseq_parse(os.fsencode(path), seq.ctypes.data_as(C.c_void_p), C.c_ulong(len(seq)),
                                lens.ctypes.data_as(C.c_void_p), C.c_ulong(len(lens)), C.byref(tot))
        assert n2 == n
        off = np.concatenate(([0], np.cumsum(lens[:n]))).astype(np.int64)
        d = K.record_digests([K.ENC[seq[off[i]:off[i + 1]]] for i in range(n)])
        seen[K.file_key(path)] = d
        return d
    K._kseq = kseq
    with tempfile.TemporaryDirectory() as tmp:
        for flavour in ("plain", "gzip", "multi", "crlf", "nofinal"):
            mp = pytest.MonkeyPatch()
            try:
                K.test_fastq_records_match_kseq(Path(tmp), mp, flavour)
            finally:
                mp.undo()
        K.test_fasta_records_match_kseq(Path(tmp))
    with open(K.GOLDEN, "w") as f:
        json.dump(seen, f, indent=0)
    print(K.GOLDEN, len(seen), "files")


def record_digamma(n=6000):
    lib = C.CDLL(os.path.join(REF, "libeigen_digamma_ref.so"))
    rng = np.random.default_rng(11)
    x = np.concatenate([10.0 ** rng.uniform(-10, 9, 40000), np.linspace(0.01, 40.0, 20000), rng.uniform(1.3, 1.6, 5000)])
    x = x[np.sort(np.random.default_rng(0).choice(len(x), n, replace=False))]
    ref = np.empty_like(x)
    lib.ref_eigen_digamma(C.c_ulong(len(x)), x.ctypes.data_as(C.c_void_p), ref.ctypes.data_as(C.c_void_p))
    out = os.path.join(HERE, "eigen_digamma.npz")
    np.savez(out, x=x, digamma=ref)
    print(out, n, "arguments")


if __name__ == "__main__":
    record_edlib()
    record_kseq()
    record_digamma()
