"""Decode conformance: edge-case and malformed streams through every decoder and entry point, checked against
the strict reference (tests/strict_ref.py).

The valid streams come from tests/edgegen.py, one family per piece of decoder code it aims at; the malformed
ones are mutants of them.  What a stream is -- valid or not, framed in 64 KiB blocks or not -- is decided by
strict_ref alone, never by how the stream was made.

CPU part: the generators, the strict reference and the oracle agree, every family hits what it aims at.
GPU part: one child process per setting of the switches the library reads once per process
(SNAPPY_B200_DECODER, SNAPPY_B200_PIECE_MIB); each decodes every stream through
every entry point and reports the calls that broke the contract as one JSON line.

Regression cases of the bugs this suite found (named by case id):
  expansion_lit1/16, expansion_copy4/17, expansion_lit4/18, expansion_mixed/20 -- valid streams longer than
      max_compressed(total) + 16 were rejected by the host calls before any kernel ran, and blocks of more than
      2 * 65536 stream bytes were reported as corrupt by the block decoders instead of going to the general decoder;
  block_reach_out/15 -- decompress_host_multi on two devices returned ERR_FRAMING for valid unframed raw Snappy;
      and k_decode_tile reported such a stream as ST_FRAMING | ST_CORRUPT (the refused copy's bytes were counted
      as missing), so the device calls gave a status that no caller can tell from a malformed stream;
  test_multi_device_forward_64mib -- SNAPPY_B200_DEVICES=2 with one usable device recursed without end.
"""
from __future__ import annotations

import json
import os
import subprocess
import sys

import numpy as np
import pytest

import edgegen
import strict_ref

BLOCK = 65536
ST_FRAMING, ST_UNRESOLVED = 4, 8
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (family, seed, total).  Totals keep streams <= 3 MiB and expansion streams <= 1 M elements; families with
# one case at <= 32 blocks and one above reach both the tile and the segment decoder under the default choice.
CASES = [
    ("seg_straddle", 1, 5 * BLOCK + 99),
    ("seg_straddle", 2, 34 * BLOCK + 7),
    ("dense", 3, 3 * BLOCK + 5),
    ("dense", 4, 34 * BLOCK),
    ("lit_threshold", 5, 4 * BLOCK + 300),
    ("literal_block", 8, 7 * BLOCK + 100),    # last block: 1 length byte
    ("literal_block", 9, 13 * BLOCK + 3000),  # 2
    ("literal_block", 10, 7 * BLOCK + 65535), # 3
    ("literal_block", 11, 40 * BLOCK + 1),    # 4, and more than 32 blocks
    ("chains_small", 12, 20 * BLOCK + 45),
    ("chains_small", 13, 3 * BLOCK + 1),
    ("block_reach", 14, 6 * BLOCK + 10),
    ("block_reach_out", 15, 5 * BLOCK + 3),
    ("expansion_lit1", 16, 200000),   # 3 stream bytes per output byte: 600 003 bytes for 200 000
    ("expansion_copy4", 17, 70000),   # copy-4 of length 1: blocks of 327 679 stream bytes
    ("expansion_lit4", 18, 100000),   # 6 stream bytes per output byte, the longest valid encoding
    ("expansion_copy2", 19, 300000),  # 1.5 per byte: longer than max_compressed, blocks still <= 2 * 65536
    ("expansion_mixed", 20, 150000),
    ("piece_edge", 21, 26 * BLOCK + 777),
]
# smaller streams of every family but piece_edge, as the bases of the mutants
MUTANT_BASES = [(f, 100 + i, (3 * BLOCK + 123) if not f.startswith("expansion") else 40000)
                for i, f in enumerate(edgegen.FAMILIES) if f != "piece_edge"]
# hand-written: the empty output with and without a trailing byte
TINY = [("empty", b"\x00"), ("empty+trailing", b"\x00\x00"), ("one-byte", b"\x01\x00a")]


def _case_id(family, seed):
    return f"{family}/{seed}"


def _max_compressed(n):
    return 10 + n + (n + BLOCK - 1) // BLOCK * 1010 if n else 0


@pytest.fixture(scope="module")
def valid_cases():
    return {_case_id(f, s): edgegen.FAMILIES[f](s, t) for f, s, t in CASES}


@pytest.fixture(scope="module")
def mutant_cases():
    """{id: (base stream, [(mutation, mutant stream)])}"""
    res = {}
    for f, s, t in MUTANT_BASES:
        stream, _ = edgegen.FAMILIES[f](s, t)
        res[_case_id(f, s)] = (stream, edgegen.mutants(stream))
    return res


# ---------------------------------------------------------------------------------------------- CPU part
def test_generators_agree_with_oracle_and_strict_reference(valid_cases, oracle):
    for cid, (stream, want) in valid_cases.items():
        assert np.array_equal(oracle.decompress(stream), want), cid
        out, why = strict_ref.strict_decode(stream)
        assert out == want.tobytes(), (cid, why)


def test_strict_layout_matches_oracle_block_index(valid_cases, mutant_cases, oracle):
    streams = [s for s, _ in valid_cases.values()] + [m for _, ms in mutant_cases.values() for _, m in ms]
    checked = 0
    for stream in streams:
        try:
            want, _ = oracle.block_index(stream)
        except ValueError:
            continue
        if strict_ref.strict_decode(stream)[0] is None:
            continue
        index, _, _ = strict_ref.strict_layout(stream)
        assert index is not None and index == [int(x) for x in want]
        checked += 1
    assert checked >= len(valid_cases)


def test_strict_reference_edges():
    """Where it is stricter than the oracle (trailing bytes, also after a declared length of 0) and the other
    rules of its docstring, on hand-written streams."""
    ok = lambda s: strict_ref.strict_decode(s)[0]
    assert ok(b"\x00") == b"" and ok(b"\x00\x00") is None
    assert ok(b"\x04\x0cabcd") == b"abcd" and ok(b"\x04\x0cabcd\x00") is None
    assert ok(b"\x08\x0cabcd" + bytes([(3 << 2) | 2, 4, 0])) == b"abcdabcd"
    assert ok(b"\x08\x0cabcd" + bytes([(3 << 2) | 2, 5, 0])) is None        # offset beyond the output
    assert ok(b"\x08\x0cabcd" + bytes([(3 << 2) | 2, 0, 0])) is None        # offset 0
    assert ok(b"\x06\x0cabcd" + bytes([(3 << 2) | 2, 1, 0])) is None        # writes past the declared length
    assert ok(b"\x04\x0cab") is None and ok(b"\x04\xf0") is None            # payload / header cut short
    assert ok(b"\x80" * 10 + b"\x00") is None                               # preamble longer than 10 bytes


def test_families_hit_their_targets(valid_cases):
    els = {cid: list(strict_ref.elements(s)) for cid, (s, _) in valid_cases.items()}

    def hdr_of(cid):
        return strict_ref.varint(valid_cases[cid][0])[1]

    # seg_straddle: tags at segment offsets 124..127 whose header crosses into the next segment, for every
    # copy header size and literal header size, and some across an 8 KiB group boundary
    for cid in ("seg_straddle/1", "seg_straddle/2"):
        h = hdr_of(cid)
        seen, group = set(), 0
        for ip, hdr, length, off, op in els[cid]:
            p = ip - h
            if p % 128 >= 124 and p % 128 + hdr > 128:
                seen.add((off is None, hdr, p % 128))
                group += (p + hdr) // 8192 != p // 8192
        for lit, hdr in [(False, 2), (False, 3), (False, 5), (True, 2), (True, 3), (True, 4), (True, 5)]:
            assert any(s[0] == lit and s[1] == hdr for s in seen), (cid, lit, hdr)
        assert {124, 125, 126, 127} <= {s[2] for s in seen}, cid
        assert group > 0, cid
    # dense: 64 element starts in one segment, two starts in one lane's 4 bytes
    h = hdr_of("dense/4")
    per_seg = np.bincount([(ip - h) // 128 for ip, *_ in els["dense/4"]])
    per_lane = np.bincount([(ip - h) // 4 for ip, *_ in els["dense/4"]])
    assert per_seg.max() == 64 and per_lane.max() == 2
    # lit_threshold: every length of LIT_LENGTHS in every legal length encoding
    got = {(length, hdr - 1) for ip, hdr, length, off, op in els["lit_threshold/5"] if off is None}
    for n in edgegen.LIT_LENGTHS:
        for k in range(5):
            if (k == 0 and n <= 60) or (k > 0 and n - 1 < 1 << (8 * k)):
                assert (n, k) in got, (n, k)
    # literal_block: one_literal_block's condition (csrc/tags.cuh) holds for whole blocks in the 2/3/4-byte
    # forms and for the last partial block with 1..4 length bytes; near misses are one byte off
    forms, last_forms, near = set(), set(), 0
    for seed in (8, 9, 10, 11):
        stream, want = valid_cases[_case_id("literal_block", seed)]
        index, _, _ = strict_ref.strict_layout(stream)
        nb = len(index) - 1
        for b in range(nb):
            c0, c1 = index[b], index[b + 1]
            olen = min(BLOCK, want.size - b * BLOCK)
            tag = int(stream[c0])
            if tag & 3 or tag >> 2 < 60:
                continue
            k = (tag >> 2) - 59
            raw = int.from_bytes(stream[c0 + 1:c0 + 1 + k].tobytes(), "little")
            if raw + 1 == olen and c1 - c0 == 1 + k + olen:
                (last_forms if b == nb - 1 and olen < BLOCK else forms).add(k)
            elif raw + 1 == olen - 1:
                near += 1
    assert forms >= {2, 3, 4} and last_forms == {1, 2, 3, 4} and near >= 2
    # chains_small: every offset 1..16 with every length 1..64, at <= 32 blocks
    pairs = {(off, length) for ip, hdr, length, off, op in els["chains_small/13"] if off is not None}
    assert {(o, n) for o in range(1, 17) for n in range(1, 65)} <= pairs
    assert valid_cases["chains_small/12"][1].size <= 32 * BLOCK
    # block_reach: sources exactly at the block's first byte (framed); one further back (not framed)
    at_start = [op for ip, hdr, length, off, op in els["block_reach/14"] if off is not None and off == op % BLOCK]
    assert len(at_start) >= 3 and strict_ref.strict_layout(valid_cases["block_reach/14"][0])[1]
    before = [op for ip, hdr, length, off, op in els["block_reach_out/15"] if off is not None and off == op % BLOCK + 1]
    assert len(before) >= 3 and not strict_ref.strict_layout(valid_cases["block_reach_out/15"][0])[1]
    # expansion: longer than max_compressed + 16, and some with blocks over 2 * 65536 stream bytes
    big_block = 0
    for cid, (stream, want) in valid_cases.items():
        if cid.startswith("expansion"):
            assert stream.size > _max_compressed(want.size) + 16, cid
            assert stream.size <= strict_ref.varint(stream)[1] + 6 * want.size
            assert len(els[cid]) <= 1 << 20
            big_block += strict_ref.strict_layout(stream)[2] > 2 * BLOCK
    assert big_block >= 3
    assert valid_cases["expansion_lit1/16"][0].size == 600003
    # piece_edge: a block starts exactly at stream offset 1 MiB
    assert (1 << 20) in strict_ref.strict_layout(valid_cases["piece_edge/21"][0])[0]


def test_mutants_have_both_verdicts(mutant_cases):
    verdicts = [strict_ref.strict_decode(m)[0] is not None for _, ms in mutant_cases.values() for _, m in ms]
    assert any(verdicts) and not all(verdicts)
    assert len(verdicts) >= 200


# ---------------------------------------------------------------------------------------------- GPU part
@pytest.fixture(scope="module")
def matrix(tmp_path_factory, valid_cases, mutant_cases):
    """Every input of the GPU children, written before any GPU call: streams in an .npz, what the strict
    reference says about them in a .json next to it."""
    arrays, meta = {}, []

    def add(cid, stream, base_index=None, cli=False):
        stream = np.frombuffer(bytes(stream), np.uint8)
        out, why = strict_ref.strict_decode(stream)
        entry = {"id": cid, "key": f"c{len(meta)}", "valid": out is not None, "why": why, "cli": cli}
        v = strict_ref.varint(stream)
        entry["total"], entry["hdr"] = (v if v else (None, None))
        if out is not None:
            index, framed, largest = strict_ref.strict_layout(stream)
            entry.update(index=index, framed=framed, largest=largest)
            arrays[entry["key"] + "w"] = np.frombuffer(out, np.uint8)
        else:
            entry.update(index=None, framed=False, largest=0)
        entry["base_index"] = base_index
        arrays[entry["key"]] = stream
        meta.append(entry)

    for cid, (stream, _) in valid_cases.items():
        add(cid, stream, cli=True)
    for name, stream in TINY:
        add(f"tiny/{name}", stream, cli=True)
    for cid, (base, muts) in mutant_cases.items():
        base_index = strict_ref.strict_layout(base)[0]
        add(cid, base, cli=True)
        for j, (name, m) in enumerate(muts):
            add(f"{cid}:{name}", m, base_index=base_index, cli=j % 5 == 0)
    d = tmp_path_factory.mktemp("conformance")
    np.savez(d / "streams.npz", **arrays)
    (d / "meta.json").write_text(json.dumps(meta))
    return d


_CHILD = r"""
import json, os, subprocess, sys, tempfile
import numpy as np, torch
sys.path.insert(0, %(root)r)
from lightweight_snappy_b200 import api
BLOCK, ST_FRAMING, ST_UNRESOLVED = 65536, 4, 8
d = sys.argv[1]
arr = np.load(os.path.join(d, "streams.npz"))
meta = json.load(open(os.path.join(d, "meta.json")))
with_cli = os.environ.get("CONFORMANCE_CLI") == "1"
two_gpus = torch.cuda.device_count() >= 2
fails = []
codecs = {}
tmp = tempfile.mkdtemp()

def codec_for(n):
    size = 1 << max(16, (max(n, 1) - 1).bit_length())
    if size not in codecs:
        codecs.clear()
        codecs[size] = api.DeviceCodec(size)
    return codecs[size]

def fail(cid, call, what):
    fails.append([cid, call, what])

def host(cid, call, fn, e, want):
    print(cid, call, flush=True)
    try:
        got = fn()
    except api.SnappyError as x:
        if e["valid"]:
            fail(cid, call, "valid stream rejected: " + str(x))
        return
    if not e["valid"]:
        fail(cid, call, "invalid stream accepted (%%d bytes out)" %% got.size)
    elif got.size != want.size or not np.array_equal(got, want):
        fail(cid, call, "wrong output")

def device(cid, e, stream, want):
    total, hdr = e["total"], e["hdr"]
    if total is None:
        return
    codec = codec_for(max(total, stream.size))
    d_stream = torch.from_numpy(np.concatenate([stream, np.zeros(64, np.uint8)])).cuda()
    out = torch.zeros(max(total, 1), dtype=torch.uint8, device="cuda")
    nb = api.block_count(total)
    fast = e["valid"] and e["index"] is not None and e["framed"] and e["largest"] <= 2 * BLOCK
    idx = e["index"] if e["valid"] else e["base_index"]
    if idx is not None and not e["valid"]:
        idx = idx[:-1] + [stream.size]
    calls = ["decompress", "async", "index"] + (["indexed"] if idx is not None and len(idx) == nb + 1 else [])
    for call in calls:
        print(cid, call, flush=True)
        out.zero_()
        offs = torch.zeros(nb + 1, dtype=torch.int64, device="cuda")
        try:
            if call == "decompress":
                codec.decompress(d_stream, stream.size, hdr, total, out, offs)
            elif call == "async":
                codec.decompress_async(d_stream, stream.size, hdr, total, out, offs, max_rounds=64)
            elif call == "index":
                if total == 0:
                    continue
                codec.index(d_stream, stream.size, hdr, total, offs)
            else:
                codec.decompress_indexed(d_stream, torch.tensor(idx, dtype=torch.int64, device="cuda"), total, out)
            torch.cuda.synchronize()
        except api.SnappyError as x:
            if e["valid"]:
                fail(cid, call, "valid stream rejected by the call: " + str(x))
            continue
        st = int(codec.status.item())
        got = out[:total].cpu().numpy()
        exact = got.size == want.size and np.array_equal(got, want) if e["valid"] else False
        if not e["valid"]:
            if st == 0 and call != "index":
                fail(cid, call, "invalid stream gave status 0")
            continue
        if call == "index":
            if st not in (0, ST_FRAMING) or (fast and st != 0):
                fail(cid, call, "status 0x%%x" %% st)
            elif st == 0 and e["index"] is not None and offs.cpu().tolist() != e["index"]:
                fail(cid, call, "K0 offsets differ from the strict index")
            continue
        ok = {0} if fast else {0, ST_FRAMING}
        if call == "async":
            ok = ok | {ST_UNRESOLVED}
        if st not in ok:
            fail(cid, call, "status 0x%%x (allowed %%s)" %% (st, sorted(ok)))
        elif st == 0 and not exact:
            fail(cid, call, "status 0 but wrong output")
        elif call == "decompress" and st == 0 and e["index"] is not None and offs.cpu().tolist() != e["index"]:
            fail(cid, call, "K0 offsets differ from the strict index")

def cli(cid, e, stream, want):
    src, dst = os.path.join(tmp, "in.snp"), os.path.join(tmp, "out.bin")
    stream.tofile(src)
    print(cid, "cli", flush=True)
    r = subprocess.run([api.CLI_PATH, "-d", src, dst], capture_output=True, text=True)
    if e["valid"] and (r.returncode != 0 or not np.array_equal(np.fromfile(dst, np.uint8), want)):
        fail(cid, "cli", "valid stream: exit %%d %%s" %% (r.returncode, r.stderr[-200:]))
    if not e["valid"] and r.returncode == 0:
        fail(cid, "cli", "invalid stream: exit 0")

canary = None
for e in meta:
    cid, stream = e["id"], arr[e["key"]]
    want = arr[e["key"] + "w"] if e["valid"] else None
    host(cid, "snappy_decompress", lambda: api.snappy_decompress(stream), e, want)
    host(cid, "host_multi(1)", lambda: api.decompress_host_multi(stream, 1), e, want)
    host(cid, "host_multi(2)", lambda: api.decompress_host_multi(stream, 2), e, want)
    idx = e["index"] if e["valid"] else e["base_index"]
    if idx is not None and e["total"] is not None and len(idx) == api.block_count(e["total"]) + 1:
        idx = np.array(idx[:-1] + [stream.size], np.uint64)
        host(cid, "host_indexed", lambda: api.decompress_host_indexed(stream, idx), e, want)
        host(cid, "host_indexed_multi(2)", lambda: api.decompress_host_multi(stream, 2, block_offsets=idx), e, want)
    if e["total"] is not None and e["total"] > 0:
        device(cid, e, stream, want)
    if with_cli and e["cli"]:
        cli(cid, e, stream, want)
    if e["valid"] and e["total"] and e["index"] is not None and e["framed"] and e["largest"] <= 2 * BLOCK:
        canary = (e, stream, want)
    elif not e["valid"] and canary is not None:
        # after a rejected stream the next valid one decodes exactly: no stale status, no stale buffers
        ce, cs, cw = canary
        host(ce["id"] + "(after " + cid + ")", "snappy_decompress", lambda: api.snappy_decompress(cs), ce, cw)
        device(ce["id"] + "(after " + cid + ")", ce, cs, cw)
print("FAILS " + json.dumps(fails))
"""

SETTINGS = {
    "auto": {},
    "seg": {"SNAPPY_B200_DECODER": "seg"},
    "tile": {"SNAPPY_B200_DECODER": "tile"},
    "pieces-1mib": {"SNAPPY_B200_PIECE_MIB": "1", "SNAPPY_B200_PIECE_START_MIB": "1"},
}
_SWITCHES = ("SNAPPY_B200_DECODER", "SNAPPY_B200_PIECE_MIB", "SNAPPY_B200_PIECE_START_MIB",
             "SNAPPY_B200_PIECE_GROWTH", "SNAPPY_B200_DEVICES")


def _run_child(code, args, env_over, timeout=900):
    env = {k: v for k, v in os.environ.items() if k not in _SWITCHES}
    env.update(env_over)
    r = subprocess.run([sys.executable, "-c", code] + args, capture_output=True, text=True, timeout=timeout, env=env)
    return r


@pytest.mark.gpu
@pytest.mark.parametrize("setting", list(SETTINGS))
def test_decode_conformance_matrix(matrix, setting):
    """Every stream through snappy_decompress, decompress_host_multi (1 and 2 devices), the indexed host calls,
    the device calls (decompress, decompress_async, decompress_indexed, index) and, under the default setting,
    `snappy_b200 -d`.  Valid streams must give exactly the strict reference's output, invalid ones an error."""
    env = dict(SETTINGS[setting])
    if setting == "auto":
        env["CONFORMANCE_CLI"] = "1"
    r = _run_child(_CHILD % {"root": ROOT}, [str(matrix)], env)
    lines = r.stdout.strip().splitlines()
    fails = [json.loads(ln[6:]) for ln in lines if ln.startswith("FAILS ")]
    assert r.returncode == 0 and fails, (f"child ended with {r.returncode}; last case: "
                                         f"{lines[-1] if lines else None}", r.stderr[-3000:])
    assert fails[0] == [], json.dumps(fails[0][:40], indent=0)


_CHILD_MULTI = r"""
import sys, numpy as np, torch
sys.path.insert(0, %(root)r); sys.path.insert(0, %(tests)r)
from lightweight_snappy_b200 import api
import edgegen, strict_ref
stream, want = edgegen.FAMILIES["block_reach_out"](15, 5 * 65536 + 3)
assert not strict_ref.strict_layout(stream)[1]
got = api.decompress_host_multi(stream, 2)
assert np.array_equal(got, want), "wrong output"
print("OK")
"""


@pytest.mark.gpu
def test_multi_device_unframed_stream():
    """decompress_host_multi over two devices on valid raw Snappy whose copies reach into earlier blocks: the
    block decoders report framing and the general decoder must take over (block_reach_out/15)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs: with one, decompress_host_multi is the one-device call")
    r = _run_child(_CHILD_MULTI % {"root": ROOT, "tests": os.path.join(ROOT, "tests")}, [], {})
    assert r.returncode == 0 and "OK" in r.stdout, (r.stdout[-2000:], r.stderr[-3000:])


_CHILD_64MIB = r"""
import sys, numpy as np
sys.path.insert(0, %(root)r); sys.path.insert(0, %(tests)r)
from lightweight_snappy_b200 import api, corpus
import oracle_lib
n = 64 << 20
data = corpus.make_corpus("mixed", n, device="cuda").cpu().numpy()
stream = oracle_lib.Oracle().compress(data, 0)
assert np.array_equal(api.snappy_decompress(stream), data), "host decode"
assert np.array_equal(api.decompress_host_multi(stream, 2), data), "multi decode"
print("OK")
"""


@pytest.mark.gpu
def test_multi_device_forward_64mib():
    """SNAPPY_B200_DEVICES=2 with one visible device: a >= 64 MiB decode is offered to the multi-device call,
    which has only one device and hands it back; that must not recurse."""
    env = {"SNAPPY_B200_DEVICES": "2", "CUDA_VISIBLE_DEVICES": os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]}
    r = _run_child(_CHILD_64MIB % {"root": ROOT, "tests": os.path.join(ROOT, "tests")}, [], env)
    assert r.returncode == 0 and "OK" in r.stdout, (r.returncode, r.stdout[-2000:], r.stderr[-3000:])
