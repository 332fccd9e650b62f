"""A strict, plain-Python reference decoder for raw Snappy, written to be read against the format.

strict_decode(stream) accepts a stream only when all of these hold:
  * the varint preamble (the declared output length) ends within 10 bytes;
  * every element header and every literal payload lies inside the stream;
  * every copy offset is in [1, bytes produced so far];
  * no element writes past the declared length;
  * the last element ends exactly at the end of the stream.

It is stricter than oracle_decompress (oracle/snappy_oracle.c) in one place: the oracle stops once the
declared length is produced and ignores whatever bytes follow, also after a declared length of 0.  The
library rejects such trailing bytes (k_decode_sequential in csrc/decode.cu ends with `ip != stream_bytes`
as an error, and the host calls check an empty stream's length up front), so this reference does too:
what it accepts is exactly what every decoder of the library must decode, and what it rejects is what
every decoder must refuse.

strict_layout(stream) describes how a valid stream sits in 64 KiB output blocks: the block index (the
stream offset at which every block starts, plus the stream length), whether every copy source lies in
the copy's own block ("framed"), and the largest block in stream bytes.
"""
from __future__ import annotations

BLOCK = 65536


def varint(stream) -> tuple[int, int] | None:
    """(declared length, preamble bytes), or None when the preamble does not end within 10 bytes."""
    stream = bytes(stream[:10])
    total = 0
    for k in range(min(len(stream), 10)):
        total |= (stream[k] & 0x7F) << (7 * k)
        if not stream[k] & 0x80:
            return total, k + 1
    return None


def header(stream, ip: int) -> tuple[int, int, int | None] | None:
    """(header bytes, output length, copy offset or None for a literal) of the element whose tag is at
    ip, or None when the header runs past the end of the stream."""
    n = len(stream)
    tag = stream[ip]
    kind = tag & 3
    if kind == 0:
        m = tag >> 2
        if m < 60:
            return 1, m + 1, None
        k = m - 59
        if ip + 1 + k > n:
            return None
        return 1 + k, int.from_bytes(bytes(stream[ip + 1:ip + 1 + k]), "little") + 1, None
    if kind == 1:
        if ip + 2 > n:
            return None
        return 2, ((tag >> 2) & 7) + 4, ((tag >> 5) << 8) | stream[ip + 1]
    size = 3 if kind == 2 else 5
    if ip + size > n:
        return None
    return size, (tag >> 2) + 1, int.from_bytes(bytes(stream[ip + 1:ip + size]), "little")


def elements(stream):
    """Yields (tag position, header bytes, output length, offset or None, output position) of a valid stream."""
    stream = bytes(stream)
    total, ip = varint(stream)
    op = 0
    while op < total:
        hdr, length, off = header(stream, ip)
        yield ip, hdr, length, off, op
        ip += hdr + (length if off is None else 0)
        op += length


def _walk(stream):
    """(output or None, reason, block index or None, framed, largest block in stream bytes)."""
    stream = bytes(stream)
    n = len(stream)
    v = varint(stream)
    if v is None:
        return None, "varint preamble does not end within 10 bytes", None, False, 0
    total, ip = v
    out = bytearray()
    index, straddles, framed = [], False, True
    while len(out) < total:
        op = len(out)
        if ip >= n:
            return None, f"stream ends at output byte {op} of {total}", None, False, 0
        if op % BLOCK == 0:
            index.append(ip)
        h = header(stream, ip)
        if h is None:
            return None, f"element header at {ip} runs past the end of the stream", None, False, 0
        hdr, length, off = h
        if op + length > total:
            return None, f"element at {ip} writes past the declared length", None, False, 0
        if op // BLOCK != (op + length - 1) // BLOCK:
            straddles = True
        if off is None:
            if ip + hdr + length > n:
                return None, f"literal at {ip} runs past the end of the stream", None, False, 0
            out += stream[ip + hdr:ip + hdr + length]
            ip += hdr + length
            continue
        if off == 0 or off > op:
            return None, f"copy at {ip} has offset {off} with {op} bytes produced", None, False, 0
        if op - off < op // BLOCK * BLOCK:
            framed = False
        src = op - off
        if off >= length:
            out += out[src:src + length]
        else:  # the copy overlaps itself: the last `off` bytes repeat
            pattern = bytes(out[src:op])
            out += (pattern * (length // off + 1))[:length]
        ip += hdr
    if ip != n:
        return None, f"{n - ip} trailing bytes after the declared length", None, False, 0
    if straddles:
        return bytes(out), "ok", None, False, 0
    index.append(n)
    largest = max((index[i + 1] - index[i] for i in range(len(index) - 1)), default=0)
    return bytes(out), "ok", index, framed, largest


def strict_decode(stream) -> tuple[bytes | None, str]:
    """(output, "ok") for a valid stream, (None, why) for an invalid one."""
    out, reason, _, _, _ = _walk(stream)
    return out, reason


def strict_layout(stream) -> tuple[list[int] | None, bool, int]:
    """For a valid stream: (block index or None when an element straddles a 64 KiB output block,
    every copy source inside its own block, largest block in stream bytes).  Raises on an invalid one."""
    out, reason, index, framed, largest = _walk(stream)
    if out is None:
        raise ValueError(reason)
    return index, framed, largest
