"""The read-file parser of the product (sb_reads_*, csrc/ingest.cu + pgzip.h) against the parser the reference tree
vendors for the same job: klibpp's kseq++ (include/kseq++.hpp).  Same files -> the same records in the same order with
the same sequence lines, for plain / gzip / concatenated-gzip FASTQ with names and comments, qualities that begin with
'@' or '+', lower case and N, CRLF line ends, a missing final newline, and single-line FASTA.  What kseq++ returns for
each generated file is stored in tests/golden/kseq_records.json, recorded from the reference's kseq++ by
tests/golden/make_ref_golden.py: the record count and a digest of every block of BLOCK records."""
import gzip
import hashlib
import json
import os

import numpy as np
import pytest

from salmon_b200 import _capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "kseq_records.json")
BLOCK = 1000

ENC = np.full(256, 4, np.uint8)
for _c, _v in zip(b"ACGTacgtUu", [0, 1, 2, 3, 0, 1, 2, 3, 3, 3]):
    ENC[_c] = _v


def file_key(path):
    """the golden file's key for a read file: the SHA-256 of its uncompressed text"""
    with open(path, "rb") as f:
        data = f.read()
    return hashlib.sha256(gzip.decompress(data) if data[:2] == b"\x1f\x8b" else data).hexdigest()


def record_digests(records):
    """the record count and, per block of BLOCK records, a digest of their lengths and 2-bit codes"""
    blocks = []
    for a in range(0, len(records), BLOCK):
        h = hashlib.sha256()
        for r in records[a:a + BLOCK]:
            h.update(len(r).to_bytes(4, "little"))
            h.update(r.tobytes())
        blocks.append(h.hexdigest()[:16])
    return {"n": len(records), "blocks": blocks}


def _kseq(path):
    """record_digests of kseq++'s records of the file at `path`, encoded with ENC, as recorded"""
    golden = json.load(open(GOLDEN))
    key = file_key(path)
    assert key in golden, "no kseq++ records recorded for this file: the generated files changed, re-record them"
    return golden[key]


def _assert_same_records(got, ref, what):
    g = record_digests(got)
    assert g["n"] == ref["n"], (what, g["n"], ref["n"])
    bad = [i for i, (x, y) in enumerate(zip(g["blocks"], ref["blocks"])) if x != y]
    assert not bad, (what, f"records {bad[0] * BLOCK} to {bad[0] * BLOCK + BLOCK - 1} differ from kseq++'s")


def _ours(path, threads, stride=320):
    got = []
    with _capi.ReadFiles(str(path), None, n_threads=threads) as rf:
        while True:
            k, left, _, ll, _ = rf.next_batch(30000, stride)
            if k == 0:
                break
            got += [left[i, :ll[i]].copy() for i in range(k)]
    return got


def _fastq(rng, n, crlf=False, final_newline=True):
    nl = b"\r\n" if crlf else b"\n"
    letters = np.frombuffer(b"ACGTNacgtn", dtype=np.uint8)
    quals = np.frombuffer(b"@+#,:FFFFFFIIII", dtype=np.uint8)
    recs = []
    for i in range(n):
        L = int(rng.integers(31, 301))
        s = letters[rng.integers(0, 4 if i % 5 else 10, L)].tobytes()
        q = quals[rng.integers(0, len(quals), L)].tobytes()
        name = b"@SRR77.%d" % i + (b" comment %d/1" % i if i % 3 else b"")
        recs.append(name + nl + s + nl + b"+" + (name[1:] if i % 7 == 0 else b"") + nl + q)
    return nl.join(recs) + (nl if final_newline else b"")


@pytest.mark.parametrize("flavour", ["plain", "gzip", "multi", "crlf", "nofinal"])
def test_fastq_records_match_kseq(tmp_path, monkeypatch, flavour):
    monkeypatch.setenv("SB_READS_INFLATERS", "3")
    monkeypatch.setenv("SB_READS_SCANNERS", "3")
    rng = np.random.default_rng({"plain": 1, "gzip": 2, "multi": 3, "crlf": 4, "nofinal": 5}[flavour])
    text = _fastq(rng, 60000, crlf=flavour == "crlf", final_newline=flavour != "nofinal")
    if flavour in ("plain", "crlf", "nofinal"):
        p = tmp_path / "r.fq"
        p.write_bytes(text)
    elif flavour == "gzip":
        p = tmp_path / "r.fq.gz"
        p.write_bytes(gzip.compress(text, 6))
    else:
        p = tmp_path / "r.fq.gz"
        step = len(text) // 4 + 1
        p.write_bytes(b"".join(gzip.compress(text[a:a + step], 5) for a in range(0, len(text), step)))
    ref = _kseq(p)
    assert ref["n"] == 60000
    for threads in (1, 8):
        _assert_same_records(_ours(p, threads), ref, (flavour, threads))


def test_fasta_records_match_kseq(tmp_path):
    rng = np.random.default_rng(9)
    letters = np.frombuffer(b"ACGTN", dtype=np.uint8)
    recs = []
    for i in range(20000):
        L = int(rng.integers(31, 301))
        recs.append(b">read%d some text\n" % i + letters[rng.integers(0, 5 if i % 9 == 0 else 4, L)].tobytes() + b"\n")
    p = tmp_path / "r.fa.gz"
    p.write_bytes(gzip.compress(b"".join(recs), 4))
    ref = _kseq(p)
    assert ref["n"] == 20000
    _assert_same_records(_ours(p, 8), ref, "fasta")
