"""CPU tests: pin the oracle (oracle/snappy_oracle.c) against the golden vectors captured
from the unmodified reference (tests/golden/golden.json) and, when the reference build is
present, against the reference itself on a fuzz set around every table-size and block
boundary (SURVEY.md section 4 / 8c)."""
import hashlib
import json
import os

import numpy as np
import pytest

import datasets

GOLDEN = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden.json")))


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.mark.parametrize("case", GOLDEN["cases"], ids=lambda c: c["spec"])
def test_oracle_matches_golden(oracle, case):
    data = datasets.gen(case["spec"])
    assert data.size == case["size"] and _sha(data) == case["input_sha256"], "input generator drifted"
    for name, mode in (("hash", 0), ("bst", 1)):
        s = oracle.compress(data, mode)
        assert s.size == case[name]["len"], name
        assert _sha(s) == case[name]["sha256"], name
        if "hex" in case[name]:
            assert s.tobytes().hex() == case[name]["hex"]
        assert np.array_equal(oracle.decompress(s), data)


def test_varint_known_answers(oracle):
    # src/test_varint.c:27-42 (127, 227, 16384) plus the reference-captured extras
    for v in GOLDEN["varints"]:
        enc = oracle.varint_encode(v["value"])
        assert enc.hex() == v["hex"]
        assert oracle.varint_decode(enc) == (v["value"], len(enc))
    assert oracle.varint_encode(127) == b"\x7f"
    assert oracle.varint_encode(227) == b"\xe3\x01"
    assert oracle.varint_encode(16384) == b"\x80\x80\x01"
    assert oracle.varint_decode(b"\x80\x80") == (0, 0)  # truncated


def test_format_example_from_slides(oracle):
    # Presentazione snappy 1/formatSnappyEx.pdf: ca 02 = 330, f0 42 = literal of 67, 09 3f = copy len 6 off 63
    assert oracle.varint_decode(b"\xca\x02") == (330, 2)
    lit = bytes(range(67))
    stream = b"\x49" + b"\xf0\x42" + lit + b"\x09\x3f"
    out = oracle.decompress(stream)
    assert out.tobytes() == lit + lit[4:10]


def test_empty_input_gives_empty_stream(oracle):
    assert oracle.compress(np.zeros(0, dtype=np.uint8), 0).size == 0
    assert oracle.compress(np.zeros(0, dtype=np.uint8), 1).size == 0


def test_decoder_accepts_copy4_and_rejects_garbage(oracle):
    # copy-4 element (src/snappy_decompression.c:323-327): literal "abcd", copy len 4 off 4
    stream = b"\x08" + b"\x0cabcd" + bytes([(3 << 2) | 3, 4, 0, 0, 0])
    assert oracle.decompress(stream).tobytes() == b"abcdabcd"
    with pytest.raises(ValueError):
        oracle.decompress(b"\x08" + b"\x0cabcd" + bytes([(3 << 2) | 2, 9, 0]))  # offset beyond output
    with pytest.raises(ValueError):
        oracle.decompress(b"\x08" + b"\x0cab")  # truncated literal


def test_block_index(oracle):
    data = datasets.gen("corpus:mixed:0:900000:200000")
    s, sizes = oracle.compress(data, 0, with_sizes=True)
    offs, total = oracle.block_index(s)
    assert total == data.size and len(offs) == 5
    hdr = len(oracle.varint_encode(data.size))
    assert offs[0] == hdr and offs[-1] == s.size
    assert np.array_equal(np.diff(offs).astype(np.uint32), sizes)


def test_oracle_vs_reference_fuzz(oracle, reference):
    specs = []
    for n in datasets.boundary_sizes():
        specs += [f"corpus:text:2:{n % 1000}:{n}", f"sym:5:{n}:{n}", f"lz:{n}:{n}", f"corpus:lowent:5:{n % 777}:{n}"]
    specs += [f"period:{p}:{p}:{n}" for p in (1, 2, 3, 5, 64, 65, 2047, 2048, 2049) for n in (4100, 66000)]
    specs += [f"corpus:random:7:0:{n}" for n in (1, 100, 65536, 65537, 140000)]
    for spec in specs:
        data = datasets.gen(spec)
        for mode in (0, 1):
            mine, theirs = oracle.compress(data, mode), reference.compress(data, mode)
            assert np.array_equal(mine, theirs), (spec, mode)
        # decoder parity: the reference decoder on the hash stream (sizes here avoid its refill bug, Q6)
        s = oracle.compress(data, 0)
        assert np.array_equal(oracle.decompress(s), data), spec
        if data.size < 131072 - 70000:
            assert np.array_equal(reference.decompress(s, data.size), data), spec


def test_reference_varint_vectors(oracle):
    theirs = {v["value"]: bytes.fromhex(v["hex"]) for v in GOLDEN["varints"]}  # captured from the reference
    for v in (0, 1, 127, 128, 227, 16384, 1 << 30, (1 << 31) - 1):
        assert oracle.varint_encode(v) == theirs[v]
        assert oracle.varint_decode(theirs[v]) == (v, len(theirs[v]))
