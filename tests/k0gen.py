"""Valid raw-Snappy streams on which K0's speculation (csrc/index.cu) fails as badly as it can.

K0 walks every 128-byte segment of the body as if an element started at its first byte and relies on those
walks merging into the true element chain; a two-level relaxation repairs the ones that do not.  The streams
here are built so that they do not merge, which makes the relaxation do all the work: one 8 KiB group per
round at worst.  Every generator is deterministic, (seed, size) -> (stream, want):

  parity_locked      every element after the first is 2 bytes long and the chain sits on odd body offsets;
                     every byte at an even offset is a copy-1 tag (byte % 4 == 1).  A walk started at an even
                     offset reads 2-byte copy-1 elements forever and never meets the chain, and the run-up of
                     k_group_init (exits of earlier segments, all even) cannot help either.
  false_kills        the same, but some even bytes are long-literal tags (0xf0 / 0xf4 / 0xf8 / 0xfc) in copy
                     offsets and literal payloads: a wrong-phase walk jumps kilobytes ahead, marks live segments
                     and groups dead and lands at a phase that depends on the bytes (dead groups keep talking,
                     the vmax bound of scatter_group).
  fake_max_literals  incompressible blocks (maximal literals "f4 ff ff" + 65 536 bytes) whose payloads all hold
                     "f4 ff ff" at the same offsets: a walk from a fake header jumps 65 539 bytes onto the next
                     fake, so chains of maximal literals run in parallel and never merge.  The stream is longer
                     than 80 % of the output, so k_group_init's literal scan runs and finds the fakes too.

Full 64 KiB blocks of the first two families are drawn from a small pool of random blocks, so that a stream of
a hundred megabytes is built in seconds; every block starts with a literal and no element straddles a block.

walk_report(stream) models the speculative walks (not the relaxation) on the CPU, to show that each family
does what it claims.  It does not predict round counts.
"""
from __future__ import annotations

import numpy as np

import strict_ref

BLOCK = 65536
SEG = 128
GROUP = 64 * SEG
MAX_LITERAL = 3 + BLOCK   # "f4 ff ff" + 65 536 bytes
FAKE_TAGS = (0xF0, 0xF4, 0xF8, 0xFC)


def varint(n: int) -> bytes:
    out = bytearray()
    while n >= 0x80:
        out.append((n & 0x7F) | 0x80)
        n >>= 7
    out.append(n)
    return bytes(out)


def ngroup_of(body_bytes: int) -> int:
    """K0's number of 8 KiB groups for a body of this many bytes."""
    return -(-body_bytes // GROUP)


def layout(stream) -> tuple[list[int], int]:
    """(block index from the strict reference, ngroup).  Raises if the stream is not valid and framed."""
    index, framed, _ = strict_ref.strict_layout(stream)
    assert index is not None and framed
    return index, ngroup_of(len(stream) - strict_ref.varint(stream)[1])


def _odd_block(rng, first: bool, max_copy_len: int, kill_p: float, body_bytes: int | None = None):
    """One block of 2-byte elements that start on odd body offsets (the block itself starts on one, except
    block 0, which opens with a 3-byte literal at offset 0).  Every byte at an even offset is = 1 (mod 4) unless
    it was turned into a fake long-literal tag (probability kill_p per element).

    body_bytes None: a full block (65 536 output bytes).  Otherwise a partial last block of exactly body_bytes
    stream bytes and fewer than 65 536 output bytes."""
    u = iter(rng.random(4 * BLOCK + 8).tolist())  # (one draw per decision: fast enough for 100 MB streams)
    pick = lambda n: int(next(u) * n)             # uniform in 0 .. n-1
    even = lambda: 4 * pick(64) + 1
    body, out = bytearray(), bytearray()
    if first:  # tag at 0 (even), payload at 1 (odd) and 2 (even)
        pay = bytes([pick(256), even()])
        body += bytes([1 << 2]) + pay
    else:
        pay = bytes([even()])
        body += bytes([0]) + pay
    out += pay
    n_out = BLOCK if body_bytes is None else BLOCK - 1
    while True:
        if body_bytes is None:
            if len(out) == n_out:
                break
            room = n_out - len(out)
        else:
            if len(body) >= body_bytes:
                break
            # every element left produces at least one byte: keep the output below one block
            room = n_out - len(out) - ((body_bytes - len(body)) // 2 - 1)
        kill = kill_p > 0 and next(u) < kill_p
        fake = FAKE_TAGS[pick(4)] if kill else None
        produced = len(out)
        if room >= 4 and next(u) < 0.95:
            length = 4 + pick(min(max_copy_len, room) - 3)
            reach = min(2047, produced)
            if fake is not None and reach >= fake:
                off = 256 * pick((reach - fake) // 256 + 1) + fake
            else:
                off = 4 * pick((reach - 1) // 4 + 1) + 1
            body += bytes([((off >> 8) << 5) | ((length - 4) << 2) | 1, off & 0xFF])
            src = produced - off
            if off >= length:
                out += out[src:src + length]
            else:  # the copy overlaps itself: the last `off` bytes repeat
                out += (bytes(out[src:]) * (length // off + 1))[:length]
        else:
            assert room >= 1
            b = fake if fake is not None else even()
            body += bytes([0, b])
            out.append(b)
    assert body_bytes is None or len(body) == body_bytes
    return bytes(body), bytes(out)


def _odd_chain(seed: int, body_bytes: int, max_copy_len: int, kill_p: float, pool: int = 16):
    assert 4 <= max_copy_len <= 11
    rng = np.random.default_rng(seed)
    target = body_bytes | 1  # block 0 opens with 3 bytes, every other element has 2: the body length is odd
    first = _odd_block(rng, True, max_copy_len, kill_p)
    if len(first[0]) + 2 > target:
        blocks = [_odd_block(rng, True, max_copy_len, kill_p, target)]
    else:
        pool = max(1, min(pool, target // len(first[0])))
        templates = [_odd_block(rng, False, max_copy_len, kill_p) for _ in range(pool)]
        blocks, size = [first], len(first[0])
        while True:
            nxt = templates[int(rng.integers(0, pool))]
            if size + len(nxt[0]) + 2 > target:
                break
            blocks.append(nxt)
            size += len(nxt[0])
        blocks.append(_odd_block(rng, False, max_copy_len, kill_p, target - size))
    want = b"".join(o for _, o in blocks)
    stream = varint(len(want)) + b"".join(b for b, _ in blocks)
    return np.frombuffer(stream, np.uint8).copy(), np.frombuffer(want, np.uint8).copy()  # (writable)


def parity_locked(seed: int, body_bytes: int, max_copy_len: int = 11):
    """A body of body_bytes (or one more: it is odd) bytes on which no speculative walk after segment 0 ever
    meets the chain.  max_copy_len=4 gives about 2 output bytes per stream byte."""
    return _odd_chain(seed, body_bytes, max_copy_len, 0.0)


def false_kills(seed: int, body_bytes: int, max_copy_len: int = 11, kill_p: float = 1 / 384):
    """parity_locked with a fake long-literal tag in the even byte of a fraction kill_p of the elements."""
    return _odd_chain(seed, body_bytes, max_copy_len, kill_p)


def fake_max_literals(seed: int, n_blocks: int, deltas=(7, 2000, 33333, 65530), last_bytes: int | None = None):
    """n_blocks - 1 incompressible 64 KiB blocks, each one maximal literal, and a last literal of last_bytes
    (257..65 535, 3-byte header) bytes.  Every payload holds "f4 ff ff" at each offset of `deltas`; in the last
    one where it fits, and no delta may leave a fake cut off by the end of the body."""
    rng = np.random.default_rng(seed)
    if last_bytes is None:
        last_bytes = int(rng.integers(257, BLOCK))
    assert n_blocks >= 1 and 257 <= last_bytes < BLOCK
    deltas = sorted(deltas)
    assert all(b - a >= 3 for a, b in zip(deltas, deltas[1:])) and deltas[-1] + 3 <= BLOCK
    assert not any(last_bytes - 3 < d < last_bytes for d in deltas), "a fake would be cut off by the end"
    want = rng.integers(0, 256, (n_blocks - 1) * BLOCK + last_bytes, dtype=np.uint8)
    fake = np.array([0xF4, 0xFF, 0xFF], np.uint8)
    for b in range(n_blocks):
        n = BLOCK if b < n_blocks - 1 else last_bytes
        for d in deltas:
            if d + 3 <= n:
                want[b * BLOCK + d:b * BLOCK + d + 3] = fake
    parts = [np.frombuffer(varint(want.size), np.uint8)]
    for b in range(n_blocks):
        n = BLOCK if b < n_blocks - 1 else last_bytes
        parts += [np.array([0xF4, (n - 1) & 0xFF, (n - 1) >> 8], np.uint8), want[b * BLOCK:b * BLOCK + n]]
    return np.concatenate(parts), want


def fake_size_for(ngroup: int) -> tuple[int, int]:
    """(n_blocks, last_bytes) of a fake_max_literals stream whose body has exactly ngroup groups."""
    for inside in (4096, 100, 8000):
        body = (ngroup - 1) * GROUP + inside
        full = max(0, (body - 3 - 1000) // MAX_LITERAL)
        last = body - 3 - full * MAX_LITERAL
        if 1000 <= last < BLOCK:
            return full + 1, last
    raise ValueError(ngroup)


# ------------------------------------------------------------------------------------------------ walk model
def _elem_size(body: np.ndarray, p: np.ndarray) -> np.ndarray:
    """Stream bytes of the element whose tag is at p, read as decode_at does (bytes past the end read 0)."""
    tag = body[p].astype(np.int64)
    kind, m = tag & 3, tag >> 2
    size = np.where(kind == 1, 2, np.where(kind == 2, 3, 5)).astype(np.int64)
    lit = kind == 0
    k = np.where(lit & (m >= 60), m - 59, 0)
    raw = np.where(lit & (m < 60), m, 0)
    for j in range(1, 5):
        raw = raw + np.where(k >= j, body[np.minimum(p + j, body.size - 1)].astype(np.int64) << (8 * (j - 1)), 0)
    return np.where(lit, 1 + k + raw + 1, size)


def chain_starts(stream) -> np.ndarray:
    """Body offsets of the true element starts (strict reference order) of a valid stream."""
    hdr = strict_ref.varint(stream)[1]
    return np.fromiter((ip - hdr for ip, *_ in strict_ref.elements(stream)), np.int64)


def walk_report(stream, starts=None, max_elems: int = 4096) -> dict:
    """Speculative walks from every 128-byte grid point of the body (or from `starts`), each followed for up to
    max_elems elements or until it meets the true chain or leaves the body.  Per walk: "merged" (met the chain),
    "steps" (elements walked), "longest" (largest element it read, in stream bytes), "end" (where it stopped)."""
    stream = np.asarray(stream, np.uint8)
    hdr = strict_ref.varint(stream)[1]
    body = np.concatenate([stream[hdr:], np.zeros(8, np.uint8)])
    n = stream.size - hdr
    on_chain = np.zeros(n + 1, bool)
    on_chain[chain_starts(stream)] = True
    p = np.arange(0, n, SEG, dtype=np.int64) if starts is None else np.asarray(starts, np.int64)
    merged = on_chain[np.minimum(p, n)] & (p < n)
    steps = np.zeros(p.size, np.int64)
    longest = np.zeros(p.size, np.int64)
    for _ in range(max_elems):
        act = np.flatnonzero(~merged & (p < n))
        if act.size == 0:
            break
        size = _elem_size(body, p[act])
        longest[act] = np.maximum(longest[act], size)
        steps[act] += 1
        p[act] += size
        inside = p[act] < n
        merged[act[inside]] = on_chain[p[act[inside]]]
    return {"start": np.arange(0, n, SEG) if starts is None else np.asarray(starts), "merged": merged,
            "steps": steps, "longest": longest, "end": p, "body": n}
