"""K0's maximal-literal cover (csrc/index.cu: k_literal_cand, k_literal_cover): incompressible 64 KiB blocks are
stored as "f4 ff ff" + 65 536 bytes, and the 8 KiB groups that lie inside such a payload are neither walked nor
resolved; they start out dead.  A candidate header q is accepted unless another candidate p shadows it
(p < q < p + 65 539).  The candidates are guesses: whatever they say, the relaxation must end on the true element
chain, so every case here is checked for exact output and for K0 block offsets equal to the strict index.

The cases:
  * mixed and random corpora at several sizes (a random stream of whole blocks ends exactly where its last
    maximal literal does);
  * a run of random blocks followed by text, with a false "f4 ff ff" planted in the run's last payload: it
    would cover text groups, and the shadow rule rejects it;
  * false "f4 ff ff" planted in text literals, some straddling group boundaries: accepted, they cover groups
    that do hold elements, which must be walked after all when the chain reaches them;
  * a lone incompressible block between compressible ones;
  * a stream cut off inside its last maximal literal, which must be refused.

literal_cover() restates the two kernels in numpy; the CPU tests check on it that each case does what it claims.
The GPU tests run the device call, the host call with 1 MiB upload pieces (so candidates meet the open end of
the bytes uploaded so far) and `snappy_b200 -d`, and check K0's round counts on larger corpora.
"""
from __future__ import annotations

import os
import subprocess

import numpy as np
import pytest

import strict_ref

BLOCK, GROUP, MAX_LITERAL = 65536, 8192, 3 + 65536
FAKE = np.array([0xF4, 0xFF, 0xFF], np.uint8)
COVERED = -1


def _corpus(kind: str, n: int, first_segment: int = 0) -> np.ndarray:
    from lightweight_snappy_b200 import corpus
    return corpus.make_corpus(kind, n, first_segment=first_segment).numpy()


def _body(stream):
    return stream[strict_ref.varint(stream)[1]:]


def literal_cover(body: np.ndarray) -> list:
    """Per group: COVERED, the offset in the group where an accepted maximal literal ends, or None."""
    n = body.size
    ngroup = -(-n // GROUP)
    pos = np.flatnonzero((body[:-2] == 0xF4) & (body[1:-1] == 0xFF) & (body[2:] == 0xFF)) if n >= 3 else []
    pos = [int(p) for p in pos if p + MAX_LITERAL <= n]
    first, last = [None] * ngroup, [None] * ngroup
    for p in pos:
        g = p // GROUP
        first[g] = p if first[g] is None else first[g]
        last[g] = p
    cands = sorted({p for p in first + last if p is not None})

    def accepted(q):
        return not any(p < q < p + MAX_LITERAL for p in cands)

    lit = [None] * ngroup
    for p in (p for p in cands if accepted(p)):
        end = p + MAX_LITERAL
        for g in range(ngroup):
            lo, hi = g * GROUP, min((g + 1) * GROUP, n)
            if first[g] is None and p + 3 <= lo and end >= hi:
                lit[g] = COVERED
            elif lo <= end < hi:
                lit[g] = end - lo
    return lit


def _starts(stream) -> np.ndarray:
    hdr = strict_ref.varint(stream)[1]
    return np.array([ip - hdr for ip, *_ in strict_ref.elements(stream)], np.int64)


def _plant_in_literals(stream, targets, shifts=(0, -1, -2)):
    """Overwrites 3 literal payload bytes with "f4 ff ff" at (or just before) each body offset in `targets`; the
    stream stays valid, only its output changes.  Returns the patched stream and the body offsets used."""
    stream = stream.copy()
    hdr = strict_ref.varint(stream)[1]
    spans = [(ip + h - hdr, ip + h - hdr + ln) for ip, h, ln, off, _ in strict_ref.elements(stream) if off is None]
    used = []
    for t in targets:
        for s in shifts:
            q = t + s
            if any(a <= q and q + 3 <= b for a, b in spans):
                stream[hdr + q:hdr + q + 3] = FAKE
                used.append(q)
                break
    return stream, used


def _make_cases(oracle) -> dict:
    cases = {}
    for kind, n in (("mixed", 3 * 2**20 + 4099), ("mixed", 5 * 2**20), ("random", 3 * 2**20 + 17),
                    ("random", 2 * 2**20)):
        want = _corpus(kind, n)
        cases[f"{kind}/{n}"] = (oracle.compress(want), want)
    # a run of random blocks, then text; a false header in the run's last payload points into the text
    rnd = _corpus("random", 3 * BLOCK)
    rnd[2 * BLOCK + 60000:2 * BLOCK + 60003] = FAKE
    want = np.concatenate([rnd, _corpus("text", 5 * BLOCK + 999)])
    cases["shadowed_fake"] = (oracle.compress(want), want)
    # false headers inside text literals, at and across group boundaries, 9 groups apart (none shadows another)
    text = oracle.compress(_corpus("text", 20 * BLOCK))
    targets = [g * GROUP + (-1, 0, 3000)[k % 3] for k, g in enumerate(range(1, _body(text).size // GROUP - 8, 9))]
    stream, _ = _plant_in_literals(text, targets)
    cases["text_fakes"] = (stream, oracle.decompress(stream))
    # one incompressible block between compressible ones
    want = np.concatenate([_corpus("text", 3 * BLOCK), _corpus("random", BLOCK), _corpus("lowent", 3 * BLOCK)])
    cases["lone_random"] = (oracle.compress(want), want)
    return cases


@pytest.fixture(scope="module")
def cases(oracle):
    return _make_cases(oracle)


@pytest.fixture(scope="module")
def truncated(oracle):
    """Two random blocks and some text, cut off 1000 bytes into the second maximal literal's payload."""
    want = np.concatenate([_corpus("random", 2 * BLOCK), _corpus("text", BLOCK)])
    stream = oracle.compress(want)
    hdr = strict_ref.varint(stream)[1]
    second = [ip for ip, h, ln, off, op in strict_ref.elements(stream) if op == BLOCK][0]
    assert bytes(stream[second:second + 3]) == b"\xf4\xff\xff"
    return stream[:second + 3 + 1000], want, hdr


# ---------------------------------------------------------------------------------------------- CPU part
def test_cases_are_valid(cases, oracle):
    for cid, (stream, want) in cases.items():
        assert np.array_equal(oracle.decompress(stream), want), cid
        index, framed, _ = strict_ref.strict_layout(stream)
        assert index is not None and framed, cid
        assert [int(x) for x in oracle.block_index(stream)[0]] == index, cid


def test_truncated_is_refused_by_the_reference(truncated):
    stream, _, _ = truncated
    assert strict_ref.strict_decode(stream)[0] is None


def test_cover_holds_no_element_on_compressor_output(cases):
    """On streams the compressor wrote, the cover is exact: random payload groups are covered, no covered
    group holds an element start, and every literal end the cover names is one."""
    for cid, (stream, _) in cases.items():
        if cid == "text_fakes":
            continue
        body, starts = _body(stream), _starts(stream)
        lit = literal_cover(body)
        start_groups = set((starts // GROUP).tolist())
        starts_set = set(starts.tolist())
        covered = [g for g, v in enumerate(lit) if v == COVERED]
        assert not start_groups & set(covered), cid
        for g, v in enumerate(lit):
            if v not in (None, COVERED):
                assert g * GROUP + v in starts_set, (cid, g)
        if cid.startswith("random"):
            # every group wholly inside a payload, except those that hold a false header
            assert len(covered) >= 0.8 * len(lit), (cid, len(covered), len(lit))


def test_shadow_rule_rejects_the_planted_header(cases):
    stream, _ = cases["shadowed_fake"]
    body, starts = _body(stream), _starts(stream)
    heads = [int(s) for s in starts if bytes(body[s:s + 3]) == b"\xf4\xff\xff"]
    assert len(heads) == 3  # the three random blocks
    fake = heads[2] + 3 + 60000
    assert bytes(body[fake:fake + 3]) == b"\xf4\xff\xff"
    text_lo = heads[2] + MAX_LITERAL
    assert fake + MAX_LITERAL > text_lo + 3 * GROUP  # accepted, it would cover text groups
    lit = literal_cover(body)
    assert all(v != COVERED for v in lit[-(-text_lo // GROUP):])
    assert lit[text_lo // GROUP] == text_lo % GROUP


def test_text_fakes_cover_live_groups(cases):
    """The planted headers are accepted and cover groups that hold elements: the GPU run must walk them."""
    stream, _ = cases["text_fakes"]
    body, starts = _body(stream), _starts(stream)
    lit = literal_cover(body)
    covered = {g for g, v in enumerate(lit) if v == COVERED}
    live_covered = covered & set((starts // GROUP).tolist())
    assert len(live_covered) >= 10
    pos = np.flatnonzero((body[:-2] == 0xF4) & (body[1:-1] == 0xFF) & (body[2:] == 0xFF))
    assert any(p % GROUP > GROUP - 3 for p in pos)  # a header that straddles a group boundary


def test_lone_random_block_is_covered(cases):
    stream, _ = cases["lone_random"]
    lit = literal_cover(_body(stream))
    assert 6 <= sum(v == COVERED for v in lit) <= 7


# ---------------------------------------------------------------------------------------------- GPU part
@pytest.mark.gpu
def test_cover_cases_through_every_entry_point(cases, truncated, tmp_path):
    import torch
    from lightweight_snappy_b200 import api

    fails = []
    for cid, (stream, want) in cases.items():
        index, _, _ = strict_ref.strict_layout(stream) if stream.size < 2**21 else (None, 0, 0)
        if index is None:
            from oracle_lib import Oracle
            index = [int(x) for x in Oracle().block_index(stream)[0]]
        total, hdr = want.size, strict_ref.varint(stream)[1]
        codec = api.DeviceCodec(max(total, stream.size))
        d_stream = torch.from_numpy(np.concatenate([stream, np.zeros(64, np.uint8)])).cuda()
        out = torch.empty(total, dtype=torch.uint8, device="cuda")
        offs = torch.zeros(api.block_count(total) + 1, dtype=torch.int64, device="cuda")
        want_index = torch.tensor(index, dtype=torch.int64, device="cuda")
        codec.decompress(d_stream, stream.size, hdr, total, out, offs)
        torch.cuda.synchronize()
        if not torch.equal(out.cpu(), torch.from_numpy(want)):
            fails.append((cid, "decompress", "output"))
        if not torch.equal(offs, want_index):
            fails.append((cid, "decompress", "block offsets"))
        offs.zero_()
        codec.index(d_stream, stream.size, hdr, total, offs)
        codec.check_status()
        if not torch.equal(offs, want_index):
            fails.append((cid, "index", "block offsets"))
        if not np.array_equal(api.snappy_decompress(stream), want):
            fails.append((cid, "snappy_decompress", "output"))
        saved = {k: os.environ.get(k) for k in ("SNAPPY_B200_PIECE_MIB", "SNAPPY_B200_PIECE_START_MIB")}
        os.environ.update({"SNAPPY_B200_PIECE_MIB": "1", "SNAPPY_B200_PIECE_START_MIB": "1"})
        try:
            if not np.array_equal(api.decompress_host(stream), want):
                fails.append((cid, "decompress_host(1 MiB pieces)", "output"))
        finally:
            for k, v in saved.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
        src, dst = tmp_path / "in.snp", tmp_path / "out.bin"
        stream.tofile(src)
        r = subprocess.run([api.CLI_PATH, "-d", str(src), str(dst)], capture_output=True, text=True)
        if r.returncode != 0 or not np.array_equal(np.fromfile(dst, np.uint8), want):
            fails.append((cid, "cli", r.returncode))
        del codec, d_stream, out
    stream, want, hdr = truncated
    with pytest.raises(api.SnappyError):
        api.snappy_decompress(stream)
    codec = api.DeviceCodec(want.size)
    d_stream = torch.from_numpy(np.concatenate([stream, np.zeros(64, np.uint8)])).cuda()
    out = torch.empty(want.size, dtype=torch.uint8, device="cuda")
    with pytest.raises(api.SnappyError):
        codec.decompress(d_stream, stream.size, hdr, want.size, out)
        codec.check_status()
    assert fails == []


@pytest.mark.gpu
def test_rounds_on_corpora():
    """With the cover, mixed data needs fewer rounds than the 11 it needed before (B200, 1 GiB: 6; 48 MiB: 4,
    text 2), and random data fewer than the 10 of the look-back scan (1 GiB: 7; 48 MiB: 5)."""
    import torch
    from lightweight_snappy_b200 import api, corpus

    n = 48 << 20
    codec = api.DeviceCodec(n)
    hdr = len(_varint(n))
    rounds = {}
    for kind in ("text", "lowent", "random", "mixed"):
        data = corpus.make_corpus(kind, n, device="cuda")
        codec.compress(data, api.MODE_HASH)
        s = codec.result_stream().clone()
        true_offs = codec.block_offsets.clone()
        offs = torch.zeros_like(true_offs)
        codec.index(s, s.numel(), hdr, n, offs)
        codec.check_status()
        rounds[kind] = api.index_rounds()
        assert torch.equal(offs, true_offs), kind
        out = torch.empty(n, dtype=torch.uint8, device="cuda")
        codec.decompress(s, s.numel(), hdr, n, out)
        codec.check_status()
        assert torch.equal(out, data), kind
    print("\nK0 rounds, 48 MiB:", rounds)
    assert rounds["mixed"] < 8, rounds
    assert rounds["random"] < 10, rounds


def _varint(n: int) -> bytes:
    out = bytearray()
    while n >= 0x80:
        out.append((n & 0x7F) | 0x80)
        n >>= 7
    out.append(n)
    return bytes(out)
