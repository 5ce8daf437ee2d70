"""The oracle's banded glocal DP recurrence (oracle/map_oracle.c dp_score -- the checker of the CUDA DP kernels) against
the reference tree's own aligner: edlib (src/edlib.cpp; salmon uses it for --recoverOrphans).  With unit costs (match 0,
mismatch -1, gap open 0, gap extend 1) the DP's best score is minus the infix (HW) edit distance of the read in the window
the band covers, as long as the band does not bind -- which holds for random sequences with a few planted edits (an
alignment that leaves the band needs more indels than the planted distance).  edlib's distances for every case these
tests generate are stored in tests/golden/edlib_hw_distance.npz, recorded from the reference's edlib build by
tests/golden/make_ref_golden.py."""
import ctypes as C
import hashlib
import os

import numpy as np

import oracle_lib as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "edlib_hw_distance.npz")


def hw_key(query: bytes, target: bytes) -> int:
    """the golden file's key for one (query, target) pair: the first 8 bytes of a SHA-256 of both"""
    return int.from_bytes(hashlib.sha256(query + b"|" + target).digest()[:8], "little")


def _edlib():
    """edlib's infix (HW) distance of a query in a target (k = -1, EDLIB_MODE_HW, EDLIB_TASK_DISTANCE), as recorded"""
    g = np.load(GOLDEN)
    dist = dict(zip(g["key"].tolist(), g["dist"].tolist()))

    def hw_distance(query: bytes, target: bytes) -> int:
        k = hw_key(query, target)
        assert k in dist, "no edlib distance recorded for this case: the generated cases changed, re-record them"
        return dist[k]
    return hw_distance


def _mutate(rng, s, n_edits):
    s = list(s)
    for _ in range(n_edits):
        kind = int(rng.integers(0, 3))
        pos = int(rng.integers(5, len(s) - 5))
        if kind == 0:
            s[pos] = (s[pos] + int(rng.integers(1, 4))) % 4
        elif kind == 1:
            s.insert(pos, int(rng.integers(0, 4)))
        else:
            del s[pos]
    return np.array(s, dtype=np.uint8)


def test_unit_cost_dp_equals_edlib_infix_distance():
    hw = _edlib()
    lib = O.load()
    lib.orc_dp_score.restype = C.c_int32
    rng = np.random.default_rng(41)
    ref = rng.integers(0, 4, 6000, dtype=np.uint8)
    ix = O.MapIndex([ref])
    p = O.map_params(ma=0, mp=-1, go=0, ge=1)
    B = p.band
    letters = np.frombuffer(b"ACGT", dtype=np.uint8)
    n_checked = 0
    for trial in range(1500):
        L = int(rng.integers(50, 151))
        start = int(rng.integers(100, len(ref) - 400))
        n_edits = int(rng.integers(0, 5))
        read = _mutate(rng, ref[start:start + L + 8], n_edits)[:L]
        ori = trial & 1
        q = read if not ori else (3 - read[::-1]).astype(np.uint8)       # what the mapper holds for a reverse-strand read
        diag = start + int(rng.integers(-3, 4))                           # the chain's diagonal is a few bases off at most
        score = lib.orc_dp_score(C.c_void_p(ix.h.value), C.byref(p), q.ctypes.data_as(C.c_void_p), C.c_uint32(L), C.c_uint32(ori),
                                 C.c_uint32(0), C.c_int32(diag))
        window = ref[max(0, diag - B): diag + L + B]
        d = hw(letters[read].tobytes(), letters[window].tobytes())
        assert d <= n_edits + 8
        assert score == -d, (trial, L, n_edits, ori, score, d)
        n_checked += 1
    assert n_checked == 1500


def test_default_scores_bound_by_edit_distance():
    """with the default scoring (ma 2, mp -4, go 6, ge 2) an alignment with e edits of the read scores at
    most ma*L (no edits) and at least ma*L - e*(ma + go + ge): edlib's distance brackets the DP score"""
    hw = _edlib()
    lib = O.load()
    lib.orc_dp_score.restype = C.c_int32
    rng = np.random.default_rng(43)
    ref = rng.integers(0, 4, 6000, dtype=np.uint8)
    ix = O.MapIndex([ref])
    p = O.map_params()
    B = p.band
    letters = np.frombuffer(b"ACGT", dtype=np.uint8)
    for trial in range(600):
        L = int(rng.integers(60, 151))
        start = int(rng.integers(100, len(ref) - 400))
        read = _mutate(rng, ref[start:start + L + 8], int(rng.integers(0, 4)))[:L]
        score = lib.orc_dp_score(C.c_void_p(ix.h.value), C.byref(p), read.ctypes.data_as(C.c_void_p), C.c_uint32(L), C.c_uint32(0),
                                 C.c_uint32(0), C.c_int32(start))
        d = hw(letters[read].tobytes(), letters[ref[max(0, start - B): start + L + B]].tobytes())
        worst_per_edit = p.ma + max(-p.mp, p.go + p.ge)
        assert p.ma * L - d * worst_per_edit <= score <= p.ma * L - (0 if d == 0 else min(-p.mp + p.ma, p.ge)), (trial, score, d, L)
        if d == 0:
            assert score == p.ma * L


def test_product_serial_dp_equals_edlib_and_oracle():
    """the product's serial DP form (map_core.h dp_score_serial, compiled for the host -- the form the warp kernel is
    checked against on the GPU): unit costs against edlib, default scoring against the oracle, same cases"""
    import hostmap_lib
    from salmon_b200._capi import map_default_params
    hw = _edlib()
    hl = hostmap_lib.build()
    hl.hmc_dp_score.restype = C.c_int32
    ol = O.load()
    ol.orc_dp_score.restype = C.c_int32
    rng = np.random.default_rng(47)
    ref = rng.integers(0, 4, 5000, dtype=np.uint8)
    off = np.array([0, len(ref)], dtype=np.uint64)
    ix = O.MapIndex([ref])
    letters = np.frombuffer(b"ACGT", dtype=np.uint8)
    pu, pd = map_default_params(ma=0, mp=-1, go=0, ge=1), map_default_params()
    ou, od = O.map_params(ma=0, mp=-1, go=0, ge=1), O.map_params(ma=pd.ma, mp=pd.mp, go=pd.go, ge=pd.ge)
    B = pu.band
    assert B == ou.band

    def prod(p, q, L, ori, diag):
        return hl.hmc_dp_score(off.ctypes.data_as(C.c_void_p), ref.ctypes.data_as(C.c_void_p), C.byref(p), q.ctypes.data_as(C.c_void_p),
                               C.c_uint32(L), C.c_uint32(ori), C.c_uint32(0), C.c_int32(diag))

    def orc(p, q, L, ori, diag):
        return ol.orc_dp_score(C.c_void_p(ix.h.value), C.byref(p), q.ctypes.data_as(C.c_void_p), C.c_uint32(L), C.c_uint32(ori),
                               C.c_uint32(0), C.c_int32(diag))
    for trial in range(1200):
        L = int(rng.integers(40, 151))
        start = int(rng.integers(100, len(ref) - 400))
        read = _mutate(rng, ref[start:start + L + 8], int(rng.integers(0, 5)))[:L]
        if trial % 9 == 0:
            read[int(rng.integers(0, L))] = 4                               # an N in the read mismatches everything
        ori = trial & 1
        q = np.ascontiguousarray(read if not ori else np.where(read[::-1] > 3, 4, 3 - read[::-1]).astype(np.uint8))
        diag = start + int(rng.integers(-3, 4))
        assert prod(pd, q, L, ori, diag) == orc(od, q, L, ori, diag), trial
        su = prod(pu, q, L, ori, diag)
        assert su == orc(ou, q, L, ori, diag), trial
        if trial % 9 != 0:
            d = hw(letters[read].tobytes(), letters[ref[max(0, diag - B): diag + L + B]].tobytes())
            assert su == -d, (trial, su, d)
    # reads that hang over either end of the reference: the DP and edlib on the clipped window agree on what is left
    for trial in range(200):
        L = 100
        over = int(rng.integers(1, 12))
        if trial & 1:
            read = np.concatenate([rng.integers(0, 4, over, dtype=np.uint8), ref[:L - over]]); diag = -over
        else:
            read = np.concatenate([ref[len(ref) - (L - over):], rng.integers(0, 4, over, dtype=np.uint8)]); diag = len(ref) - (L - over)
        q = np.ascontiguousarray(read)
        assert prod(pd, q, L, 0, diag) == orc(od, q, L, 0, diag), trial
        assert prod(pu, q, L, 0, diag) == orc(ou, q, L, 0, diag), trial
