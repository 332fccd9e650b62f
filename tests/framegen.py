"""The Snappy framing format (google/snappy framing_format.txt) in plain Python, written to be read against it.

  crc32c / masked_crc      CRC-32C (Castagnoli, reflected 0x82F63B78, init and final xor 0xffffffff) and its mask
  frame_compress_ref       the writer rule of include/snappy_b200.h on top of the CPU oracle's raw compressor:
                           identifier, then one chunk per 64 KiB block, compressed (0x00) when varint(n) + the block's
                           elements is shorter than n - n // 8, uncompressed (0x01) otherwise
  unframe                  a strict unframer, the arbiter of valid / corrupt / checksum for framed streams as
                           strict_ref.py is for raw streams: every header rule first, then every payload (a raw
                           Snappy buffer that strict_decode accepts, declaring at most 65536 bytes), then every CRC
  foreign_streams          deterministic valid streams in shapes our writer does not emit
  mutants                  malformed or mis-checksummed variants of a valid stream
"""
from __future__ import annotations

import numpy as np

from strict_ref import strict_decode

BLOCK = 65536
STREAM_ID = b"\xff\x06\x00\x00sNaPpY"
POLY = 0x82F63B78

_T = np.zeros(256, dtype=np.uint32)
for _i in range(256):
    _c = _i
    for _ in range(8):
        _c = (_c >> 1) ^ POLY if _c & 1 else _c >> 1
    _T[_i] = _c
_TL = [int(x) for x in _T]


def crc32c_bitwise(data) -> int:
    c = 0xFFFFFFFF
    for x in bytes(data):
        c ^= x
        for _ in range(8):
            c = (c >> 1) ^ POLY if c & 1 else c >> 1
    return c ^ 0xFFFFFFFF


def crc32c(data) -> int:
    c = 0xFFFFFFFF
    for x in bytes(data):
        c = (c >> 8) ^ _TL[(c ^ x) & 0xFF]
    return c ^ 0xFFFFFFFF


def _crc32c_rows(m: np.ndarray) -> np.ndarray:
    """CRC-32C of every row of a 2-D uint8 array (the rows are processed side by side)."""
    c = np.full(m.shape[0], 0xFFFFFFFF, dtype=np.uint32)
    for j in range(m.shape[1]):
        c = (c >> np.uint32(8)) ^ _T[(c ^ m[:, j]) & np.uint32(0xFF)]
    return c ^ np.uint32(0xFFFFFFFF)


def block_crcs(data: np.ndarray) -> list[int]:
    """CRC-32C of every 64 KiB block of data (the last one may be shorter)."""
    data = np.ascontiguousarray(data, dtype=np.uint8)
    full = data.size // BLOCK
    res = [int(x) for x in _crc32c_rows(data[: full * BLOCK].reshape(full, BLOCK))] if full else []
    if data.size % BLOCK:
        res.append(crc32c(data[full * BLOCK:].tobytes()))
    return res


def mask(c: int) -> int:
    return (((c >> 15) | (c << 17)) + 0xA282EAD8) & 0xFFFFFFFF


def masked_crc(data) -> int:
    return mask(crc32c(data))


def varint(n: int) -> bytes:
    out = bytearray()
    while n >= 0x80:
        out.append((n & 0x7F) | 0x80)
        n >>= 7
    out.append(n)
    return bytes(out)


def chunk(ctype: int, payload: bytes) -> bytes:
    return bytes([ctype]) + len(payload).to_bytes(3, "little") + payload


def data_chunk(raw: bytes, snappy_payload: bytes | None = None, crc: int | None = None) -> bytes:
    """A compressed chunk when snappy_payload (varint(n) || elements) is given, an uncompressed one otherwise."""
    c = (masked_crc(raw) if crc is None else crc).to_bytes(4, "little")
    return chunk(0x00, c + snappy_payload) if snappy_payload is not None else chunk(0x01, c + bytes(raw))


# ---------------------------------------------------------------------------------------------- the writer
def frame_compress_ref(oracle, data, mode: int = 0, identifier: bool = True) -> bytes:
    """What the library's framed compressor must write.  The oracle compresses every block on its own tables,
    so block b's elements in the oracle's raw stream are exactly those of compressing block b alone."""
    data = np.ascontiguousarray(data, dtype=np.uint8)
    parts = [STREAM_ID] if identifier else []
    if data.size == 0:
        return b"".join(parts)
    raw, sizes = oracle.compress(data, mode, with_sizes=True)
    raw = raw.tobytes()
    pos = len(varint(data.size))
    for b, crc in enumerate(block_crcs(data)):
        blk = data[b * BLOCK:(b + 1) * BLOCK].tobytes()
        n, s = len(blk), int(sizes[b])
        elems = raw[pos:pos + s]
        pos += s
        payload = varint(n) + elems
        parts.append(data_chunk(blk, payload if len(payload) < n - n // 8 else None, mask(crc)))
    assert pos == len(raw)
    return b"".join(parts)


# ---------------------------------------------------------------------------------------------- the arbiter
def walk(stream) -> tuple[list[tuple[int, int, int, bytes]] | None, str]:
    """Header rules only: ([(offset, type, masked crc, body)] of the data chunks, 'ok') or (None, 'corrupt').
    For a compressed chunk the body is the whole raw Snappy buffer, varint included."""
    s = bytes(stream)
    if not s:
        return [], "ok"
    if s[:10] != STREAM_ID:
        return None, "corrupt"
    at, res = 10, []
    while at < len(s):
        if len(s) - at < 4:
            return None, "corrupt"
        t, L = s[at], int.from_bytes(s[at + 1:at + 4], "little")
        if L > len(s) - at - 4:
            return None, "corrupt"
        body = s[at + 4:at + 4 + L]
        if t in (0x00, 0x01):
            if L < 4:
                return None, "corrupt"
            if t == 0x00:
                n = 0
                for k in range(min(L - 4, 10) + 1):
                    if k == min(L - 4, 10):
                        return None, "corrupt"  # the varint does not end inside the chunk
                    n |= (body[4 + k] & 0x7F) << (7 * k)
                    if not body[4 + k] & 0x80:
                        break
                if n > BLOCK:
                    return None, "corrupt"
            elif L - 4 > BLOCK:
                return None, "corrupt"
            res.append((at, t, int.from_bytes(body[:4], "little"), body[4:]))
        elif t == 0xFF:
            if body != STREAM_ID[4:]:
                return None, "corrupt"
        elif t < 0x80:
            return None, "corrupt"
        at += 4 + L
    return res, "ok"


def unframe(stream) -> tuple[bytes | None, str]:
    """(data, 'ok'), or (None, 'corrupt' | 'checksum'): malformed anywhere wins over a checksum mismatch."""
    chunks, verdict = walk(stream)
    if chunks is None:
        return None, verdict
    outs = []
    for _, t, _, body in chunks:
        if t == 0x01:
            outs.append(body)
            continue
        out, _ = strict_decode(body)
        if out is None:
            return None, "corrupt"
        outs.append(out)
    if any(mask(crc32c(o)) != c for o, (_, _, c, _) in zip(outs, chunks)):
        return None, "checksum"
    return b"".join(outs), "ok"


def total_length(stream) -> int | None:
    chunks, _ = walk(stream)
    if chunks is None:
        return None
    total = 0
    for _, t, _, body in chunks:
        if t == 0x01:
            total += len(body)
        else:
            n, k = 0, 0
            while True:
                n |= (body[k] & 0x7F) << (7 * k)
                if not body[k] & 0x80:
                    break
                k += 1
            total += n
    return total


# ---------------------------------------------------------------------------------------------- generators
EDGE_FAMILIES = ("expansion_copy4", "expansion_lit4", "expansion_mixed", "lit_threshold", "literal_block", "dense",
                 "chains_small")


def foreign_streams(oracle) -> list[tuple[str, bytes, bytes]]:
    """(name, stream, data): chunk sizes 0..65536, padding and skippable chunks, repeated identifiers, and
    compressed payloads no block compressor emits (tests/edgegen.py families of at most 65536 output bytes:
    copy-4, 4-byte literal lengths, long literals, 6x expansion -- a body past 2 * 65536 bytes)."""
    import edgegen
    rng = np.random.default_rng(2024)
    res = []

    def add(name, pieces):
        stream = STREAM_ID + b"".join(p[0] for p in pieces)
        res.append((name, stream, b"".join(p[1] for p in pieces)))

    def comp(raw):  # (the oracle writes nothing at all for an empty input; a chunk's buffer is varint(0) then)
        payload = oracle.compress(np.frombuffer(raw, np.uint8), 0).tobytes() if raw else b"\x00"
        return data_chunk(raw, payload), raw

    def unc(raw):
        return data_chunk(raw), raw

    text = bytes(rng.integers(97, 101, 3 * BLOCK, dtype=np.uint8))
    rnd = bytes(rng.integers(0, 256, 2 * BLOCK, dtype=np.uint8))
    for n in (0, 1, 2, 100, 4095, 65535, 65536):
        add(f"compressed-{n}", [comp(text[:n])])
        add(f"uncompressed-{n}", [unc(rnd[:n])])
    add("empty-compressed-only", [(data_chunk(b"", b"\x00"), b"")])
    add("empty-uncompressed-only", [(data_chunk(b""), b"")])
    add("identifier-only", [])
    pad = (chunk(0xFE, bytes(37)), b"")
    skip = (chunk(0x80, b"skip me"), b"")
    skip2 = (chunk(0xFD, bytes(300)), b"")
    empty_skip = (chunk(0x99, b""), b"")
    again = (STREAM_ID, b"")
    add("mixed-sizes", [comp(text[:300]), unc(rnd[:7]), comp(text[300:300 + BLOCK]), pad, unc(rnd[:BLOCK]),
                        again, comp(b""), skip, unc(b""), comp(text[:12345]), skip2, empty_skip])
    add("leading-padding", [pad, again, comp(text[:5000]), unc(rnd[:5000])])
    add("many-small", [comp(text[i:i + 1 + i % 97]) if i % 3 else unc(rnd[i:i + i % 131]) for i in range(0, 600, 7)])
    for name in EDGE_FAMILIES:
        for total in (1000, BLOCK):
            s, d = edgegen.FAMILIES[name](7, total)
            add(f"edge-{name}-{total}", [(data_chunk(d.tobytes(), s.tobytes()), d.tobytes()), unc(rnd[:99])])
    return res


def mutants(stream) -> list[tuple[str, bytes]]:
    """Malformed or mis-checksummed variants of a valid framed stream with at least one data chunk.  Whether a
    mutant is corrupt or only fails its checksum is for unframe() to say, not for its name."""
    s = bytes(stream)
    chunks, _ = walk(s)
    assert chunks
    res = [("no-identifier", s[10:]), ("identifier-altered", s[:6] + bytes([s[6] ^ 0x20]) + s[7:]),
           ("identifier-short", s[:9]), ("unskippable-0x02", s + chunk(0x02, b"xy")),
           ("unskippable-0x7f", s[:10] + chunk(0x7F, b"") + s[10:]),
           ("bad-repeat-identifier", s + chunk(0xFF, b"sNaPpy")),
           ("n>65536", s + chunk(0x00, mask(0).to_bytes(4, "little") + varint(BLOCK + 1) + b"\x00")),
           ("uncompressed>65536", s + data_chunk(bytes(BLOCK + 1))),
           ("crc-only-chunk", s + chunk(0x01, b"\x00\x00\x00")),
           ("bad-varint", s + chunk(0x00, bytes(4) + b"\x80\x80"))]
    last_at, t, crc, body = chunks[-1]
    end = last_at + 4 + 4 + len(body)
    res += [("truncated-header", s[:last_at + 2]), ("truncated-payload", s[:end - 1] if len(body) else s[:end - 3]),
            ("length-past-end", s[:last_at + 1] + (len(body) + 5).to_bytes(3, "little") + s[last_at + 4:]),
            ("trailing-garbage", s + b"\x00\x01\x02")]
    for at, t, crc, body in chunks[:1] + chunks[len(chunks) // 2:len(chunks) // 2 + 1]:
        h = at + 4
        res.append((f"crc-flip@{at}", s[:h + 1] + bytes([s[h + 1] ^ 0x10]) + s[h + 2:]))
        if body:
            i = h + 4 + len(body) - 1  # the chunk's last byte: a data byte, or (compressed) usually a literal's
            res.append((f"data-flip@{at}", s[:i] + bytes([s[i] ^ 0x01]) + s[i + 1:]))
        # one more byte inside the chunk: trailing bytes after the buffer, or one more data byte
        L = 4 + len(body) + 1
        res.append((f"trailing-byte@{at}", s[:at] + bytes([t]) + L.to_bytes(3, "little") + s[h:h + 4 + len(body)] +
                    b"\x00" + s[h + 4 + len(body):]))
    return res
