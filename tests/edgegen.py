"""Valid raw-Snappy streams built to sit on the edges of the decoders, and malformed mutants of them.

Every family is a deterministic (seed, total) -> (stream, want) and aims at one piece of the library:

  seg_straddle   element headers that start at 128-byte segment offsets 124..127 and cross into the next
                 segment (2/3/5-byte copy headers, 2..5-byte literal headers), also across 8 KiB groups:
                 K0's walks and maps (csrc/index.cu), k_decode_seg's start-map masking, the tile staging halo
  dense          runs of copy-1 elements (2 bytes): 64 element starts in one segment, two in one lane's 4 bytes
  lit_threshold  literals of 1, 59..65 and 255..257 bytes in every legal length encoding: the long-literal
                 threshold (kLongLiteral) and the 5-byte-header path
  literal_block  blocks that are one literal in the 2/3/4-byte length forms, a last partial block that is one
                 literal with 1..4 length bytes, and near misses: one_literal_block, k_copy_literal_blocks and
                 the tile decoder's single-literal fast path
  chains_small   short overlapping copy chains at <= 32 blocks, and every offset 1..16 with every length 1..64:
                 k_decode_tile's phase C and do_copy, k_decode_warp on the indexed path
  block_reach    copies whose source is exactly the first byte of their block (framed)
  block_reach_out  ... and copies whose offset is one larger (valid raw Snappy, not framed)
  expansion_*    streams far longer than max_compressed of their output (1-byte literals with 2..5-byte headers,
                 copy-2 / copy-4 of length 1..3): the host length pre-checks and blocks > 2 * 65536 stream bytes
  piece_edge     a block boundary exactly on a 1 MiB stream offset, where the host pipeline cuts an upload piece
                 under SNAPPY_B200_PIECE_MIB=1

Streams never let an element straddle a 64 KiB output block.  Apart from block_reach_out they are framed.
"""
from __future__ import annotations

import numpy as np

BLOCK = 65536
SEG = 128
GROUP = 64 * SEG


def varint(n: int) -> bytes:
    out = bytearray()
    while n >= 0x80:
        out.append((n & 0x7F) | 0x80)
        n >>= 7
    out.append(n)
    return bytes(out)


def lit_header(n: int, k: int) -> bytes:
    """Header of an n-byte literal with k length bytes (k = 0: the length in the tag, n <= 60)."""
    if k == 0:
        assert 1 <= n <= 60
        return bytes([(n - 1) << 2])
    assert n - 1 < 1 << (8 * k)
    return bytes([(59 + k) << 2]) + (n - 1).to_bytes(k, "little")


def copy_elem(length: int, off: int, size: int) -> bytes:
    """A copy with a `size`-byte header: 2 (copy-1), 3 (copy-2) or 5 (copy-4)."""
    if size == 2:
        assert 4 <= length <= 11 and off < 2048
        return bytes([((off >> 8) << 5) | ((length - 4) << 2) | 1, off & 0xFF])
    assert 1 <= length <= 64
    if size == 3:
        return bytes([((length - 1) << 2) | 2]) + off.to_bytes(2, "little")
    return bytes([((length - 1) << 2) | 3]) + off.to_bytes(4, "little")


class Writer:
    """Appends elements and keeps the expected output.  Positions are body-relative (after the varint),
    which is how K0 cuts the stream into 128-byte segments."""

    def __init__(self, seed: int, total: int):
        self.rng = np.random.default_rng(seed)
        self.total = total
        self.head = varint(total)
        self.body = bytearray()
        self.out = bytearray()

    @property
    def pos(self) -> int:
        return len(self.body)

    @property
    def done(self) -> int:  # output bytes produced in the current block
        return len(self.out) % BLOCK

    @property
    def room(self) -> int:  # output bytes left in the current block
        return min(BLOCK - self.done, self.total - len(self.out))

    def lit(self, n: int, k: int | None = None) -> None:
        if k is None:
            k = 0 if n <= 60 else (1 if n <= 256 else 2)
        data = self.rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        self.body += lit_header(n, k) + data
        self.out += data

    def copy(self, length: int, off: int, size: int) -> None:
        self.body += copy_elem(length, off, size)
        start = len(self.out) - off
        for i in range(length):
            self.out.append(self.out[start + i])

    def filler(self, nbytes: int) -> None:
        """One element of exactly nbytes (2 or 3) stream bytes: a 1- or 2-byte literal, or a 1-byte
        literal with a 1-byte length when only one output byte is left in the block."""
        if nbytes == 2:
            self.lit(1, 0)
        elif self.room >= 2:
            self.lit(2, 0)
        else:
            self.lit(1, 1)

    def pad_to(self, target: int) -> None:
        """Fillers until the next tag is at body position target (target - pos must be 0 or >= 2)."""
        while self.pos < target and self.room:
            d = target - self.pos
            self.filler(3 if d % 2 else 2)

    def ordinary(self) -> None:
        """A random element that fits the block: a short literal, or a copy within the block."""
        room, done = self.room, self.done
        if done == 0 or self.rng.random() < 0.3:
            self.lit(int(self.rng.integers(1, min(room, 80) + 1)))
            return
        off = int(self.rng.integers(1, min(done, 2047) + 1))
        if room >= 4 and self.rng.random() < 0.5:
            self.copy(int(self.rng.integers(4, min(room, 11) + 1)), off, 2)
        else:
            self.copy(int(self.rng.integers(1, min(room, 64) + 1)), off, 3)

    def result(self) -> tuple[np.ndarray, np.ndarray]:
        assert len(self.out) == self.total, (len(self.out), self.total)
        stream = self.head + bytes(self.body)
        return np.frombuffer(stream, np.uint8).copy(), np.frombuffer(bytes(self.out), np.uint8).copy()


# ---------------------------------------------------------------------------------------------- families
def seg_straddle(seed: int, total: int):
    """Every few segments: a tag at segment offset 124..127 whose header crosses into the next segment."""
    w = Writer(seed, total)
    kinds = [("copy", 2), ("copy", 3), ("copy", 5), ("lit", 1), ("lit", 2), ("lit", 3), ("lit", 4)]
    j = 0
    while w.room:
        w.ordinary()
        if not w.room:
            break
        # the next segment boundary at least 8 bytes ahead (every 64th one is an 8 KiB group boundary)
        boundary = (w.pos + 8 + SEG - 1) // SEG * SEG
        kind, size = kinds[j % len(kinds)]
        hdr = size if kind == "copy" else size + 1
        r = 1 + (j // len(kinds)) % min(hdr - 1, 4)  # the tag sits r bytes before the boundary
        w.pad_to(boundary - r)
        if not w.room:
            break
        if kind == "copy" and w.done > 0 and (size != 2 or w.room >= 4):
            off = int(w.rng.integers(1, min(w.done, 2047) + 1))
            w.copy(4 if size == 2 else int(w.rng.integers(1, min(w.room, 64) + 1)), off, size)
        elif kind == "lit":
            w.lit(int(w.rng.integers(1, min(w.room, 100) + 1)), size)
        j += 1
    return w.result()


def dense(seed: int, total: int):
    """Blocks of copy-1 elements only (2 stream bytes each) after an opening literal of even size."""
    w = Writer(seed, total)
    while w.room:
        if w.done == 0:
            w.lit(min(w.room, 15), 0)  # 16 stream bytes: the copies stay on even positions
        elif w.room >= 4:
            w.copy(int(w.rng.integers(4, min(w.room, 11) + 1)), int(w.rng.integers(1, min(w.done, 2047) + 1)), 2)
        else:
            w.lit(1, 0)
    return w.result()


LIT_LENGTHS = [1] + list(range(59, 66)) + [255, 256, 257]


def lit_threshold(seed: int, total: int):
    """Every literal length of LIT_LENGTHS in every legal length encoding, between ordinary elements."""
    w = Writer(seed, total)
    combos = [(n, k) for n in LIT_LENGTHS for k in range(5) if (k == 0 and n <= 60) or (k > 0 and n - 1 < 1 << (8 * k))]
    j = 0
    while w.room:
        n, k = combos[j % len(combos)]
        if n <= w.room:
            w.lit(n, k)
            j += 1
        if w.room:
            w.ordinary()
    return w.result()


def literal_block(seed: int, total: int):
    """Whole blocks as one literal (2, 3 and 4 length bytes), near misses, ordinary blocks, and a last
    partial block that is one literal with 1 + seed % 4 length bytes (1 only when it is <= 256 bytes)."""
    w = Writer(seed, total)
    b = 0
    while w.room:
        if w.room < BLOCK:  # the last, partial block
            k = 1 + seed % 4
            if w.room > 256 and k == 1:
                k = 2
            w.lit(w.room, k)
            break
        kind = b % 6
        if kind < 3:
            w.lit(BLOCK, 2 + kind)
        elif kind == 3:  # 65535-byte literal + a 1-byte literal
            w.lit(BLOCK - 1, 2)
            w.lit(1, 0)
        elif kind == 4:  # 65535-byte literal + a copy of length 1
            w.lit(BLOCK - 1, 3)
            w.copy(1, int(w.rng.integers(1, 1000)), 3)
        else:
            w.ordinary()
            while w.done:
                w.ordinary()
        b += 1
    return w.result()


def chains_small(seed: int, total: int):
    """Every offset 1..16 with every length 1..64 (copy-2) in the first block, then chains of short
    overlapping copies (offsets 1..40, lengths 4..64) cut now and then by literals and copy-4s."""
    w = Writer(seed, total)
    w.lit(min(w.room, 16), 0)
    for off in range(1, 17):
        for length in range(1, 65):
            if w.room < length:
                break
            w.copy(length, off, 3)
    while w.room:
        if w.done == 0 or w.rng.random() < 0.1:
            w.lit(int(w.rng.integers(1, min(w.room, 17) + 1)))
            continue
        if w.rng.random() < 0.03:
            w.lit(min(w.room, int(w.rng.integers(64, 300))))
            continue
        length = min(int(w.rng.integers(4, 65)), w.room)
        off = int(w.rng.integers(1, min(w.done, 40) + 1))
        size = 5 if w.rng.random() < 0.05 else (2 if 4 <= length <= 11 else 3)
        w.copy(length, off, size)
    return w.result()


def _block_reach(seed: int, total: int, extra: int):
    """Copies with offset = (bytes produced in the block) + extra, of every header size, a few per block."""
    w = Writer(seed, total)
    j = 0
    while w.room:
        w.ordinary()
        if w.room and w.done and (len(w.out) >= BLOCK or extra == 0) and w.rng.random() < 0.2:
            off = w.done + extra
            size = (2, 3, 5)[j % 3]
            if size == 2 and (off >= 2048 or w.room < 4):
                size = 3
            if size == 3 and off > 0xFFFF:
                size = 5
            length = 4 if size == 2 else int(w.rng.integers(1, min(w.room, 64) + 1))
            w.copy(length, off, size)
            j += 1
    return w.result()


def block_reach(seed: int, total: int):
    return _block_reach(seed, total, 0)


def block_reach_out(seed: int, total: int):
    return _block_reach(seed, total, 1)


def _expansion(seed: int, total: int, form: str):
    """Output written one to three bytes per element in a wasteful form:
    'lit1' 1-byte literals with a 1-byte length (3 stream bytes per output byte), 'lit4' with a 4-byte
    length (6 per byte), 'copy4' copy-4 of length 1 (5 per byte), 'copy2' copy-2 of length 2 (1.5 per byte),
    'mixed' 1-byte literals with 1..4 length bytes, copy-4 of length 1 and copy-2 of length 1..3."""
    w = Writer(seed, total)
    while w.room:
        f = form if form != "mixed" else ("lit1", "lit2", "lit3", "lit4", "copy4", "copy2s")[int(w.rng.integers(0, 6))]
        if f.startswith("lit") or w.done == 0:
            k = int(f[3]) if f.startswith("lit") else 2
            w.lit(1, k)
        elif f == "copy4":
            w.copy(1, int(w.rng.integers(1, w.done + 1)), 5)
        elif f == "copy2":
            w.copy(min(2, w.room), int(w.rng.integers(1, w.done + 1)), 3)
        else:
            w.copy(min(int(w.rng.integers(1, 4)), w.room), int(w.rng.integers(1, w.done + 1)), 3)
    return w.result()


def piece_edge(seed: int, total: int):
    """Ordinary blocks until the stream nears 1 MiB, then a block of literals whose stream size puts the
    next block's first tag exactly at stream offset 1 MiB, then ordinary blocks again."""
    w = Writer(seed, total)
    edge = (1 << 20) - len(w.head)  # body-relative
    placed = False
    while w.room:
        left = edge - w.pos
        if not placed and w.done == 0 and left <= 2 * BLOCK + 3:
            assert left >= BLOCK + 3 and w.room == BLOCK
            n1 = left - (BLOCK + 3)  # 1-byte literals (2 stream bytes each), then one literal of the rest
            for _ in range(n1):
                w.lit(1, 0)
            w.lit(BLOCK - n1, 2)
            assert w.pos == edge
            placed = True
            continue
        if w.done == 0 and not placed:  # half literal, half copies: about 34 KiB of stream per block
            w.lit(BLOCK // 2, 2)
            continue
        w.ordinary()
    assert placed
    return w.result()


FAMILIES = {
    "seg_straddle": seg_straddle,
    "dense": dense,
    "lit_threshold": lit_threshold,
    "literal_block": literal_block,
    "chains_small": chains_small,
    "block_reach": block_reach,
    "block_reach_out": block_reach_out,
    "expansion_lit1": lambda seed, total: _expansion(seed, total, "lit1"),
    "expansion_lit4": lambda seed, total: _expansion(seed, total, "lit4"),
    "expansion_copy4": lambda seed, total: _expansion(seed, total, "copy4"),
    "expansion_copy2": lambda seed, total: _expansion(seed, total, "copy2"),
    "expansion_mixed": lambda seed, total: _expansion(seed, total, "mixed"),
    "piece_edge": piece_edge,
}


# ---------------------------------------------------------------------------------------------- mutants
def _with_varint(stream: bytes, total: int) -> bytes:
    from strict_ref import varint as parse
    _, hdr = parse(stream)
    return varint(total) + stream[hdr:]


def mutants(stream) -> list[tuple[str, bytes]]:
    """(name, mutated stream) at chosen elements of a valid stream: the first element, one in the middle of
    a middle block, the last one of the first block, and the last one overall.  Whether a mutant is valid is
    for the strict reference to say, not for its name."""
    from strict_ref import elements, varint as parse
    stream = bytes(stream)
    total, _ = parse(stream)
    els = list(elements(stream))
    if not els:
        return []
    nb = (total + BLOCK - 1) // BLOCK
    mid_blk = nb // 2
    in_mid = [e for e in els if e[4] // BLOCK == mid_blk]
    in_first = [e for e in els if e[4] < BLOCK]
    chosen = {"first": els[0], "mid": in_mid[len(in_mid) // 2], "blockend": in_first[-1], "last": els[-1]}
    res = [("append", stream + b"\x00"), ("declared-1", _with_varint(stream, total - 1)),
           ("declared+1", _with_varint(stream, total + 1)), ("declared+65536", _with_varint(stream, total + BLOCK))]
    for where, (ip, hdr, length, off, op) in chosen.items():
        tag = stream[ip]
        res.append((f"{where}:cut", stream[:ip]))
        res.append((f"{where}:cut+1", stream[:ip + 1]))
        res.append((f"{where}:type^1", stream[:ip] + bytes([tag ^ 1]) + stream[ip + 1:]))
        res.append((f"{where}:type^2", stream[:ip] + bytes([tag ^ 2]) + stream[ip + 1:]))
        if off is not None:
            if hdr == 2:
                enc = lambda o: bytes([(tag & 0x1F) | ((o >> 8) << 5), o & 0xFF]) if o < 2048 else None
            else:
                enc = lambda o: bytes([tag]) + o.to_bytes(hdr - 1, "little") if o < 1 << (8 * (hdr - 1)) else None
            for name, o in (("off0", 0), ("off=produced+1", op + 1)):
                e = enc(o)
                if e is not None:
                    res.append((f"{where}:{name}", stream[:ip] + e + stream[ip + hdr:]))
        else:
            m = tag >> 2
            if m < 59:  # in the tag: one more (a tag of 60 would mean "one length byte follows")
                res.append((f"{where}:len+1", stream[:ip] + bytes([tag + 4]) + stream[ip + 1:]))
                res.append((f"{where}:len=ones", stream[:ip] + bytes([59 << 2]) + stream[ip + 1:]))
            elif m >= 60:
                k = m - 59
                if length < 1 << (8 * k):
                    res.append((f"{where}:len+1", stream[:ip + 1] + length.to_bytes(k, "little") + stream[ip + 1 + k:]))
                res.append((f"{where}:len=ones", stream[:ip + 1] + b"\xff" * k + stream[ip + 1 + k:]))
    return res
