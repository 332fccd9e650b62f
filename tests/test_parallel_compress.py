"""SNAPPY_B200_MODE_PARALLEL: the block-parallel parse.

Its stream is valid Snappy in the reference's format but not the reference's bytes, so what it must be is
defined by a CPU model (tests/parallel_parse.c, built here with the constants of csrc/parallel_parse.h).
The CPU tests hold the model to the stream invariants the decoders rely on and to its size targets; the GPU
tests hold every compress entry point to the model byte for byte and run the streams through every decoder.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import datasets
import framegen
import strict_ref
from lightweight_snappy_b200 import api, corpus

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BLOCK = 65536
SLICE = 2048
MAX_BLOCK_BYTES = BLOCK + 1010
MODE_PARALLEL = 2


# ---------------------------------------------------------------------------------------------- the model
class ParallelModel:
    def __init__(self, so_path: str):
        L = C.CDLL(so_path)
        L.oracle_compress_parallel.restype = C.c_uint64
        L.oracle_compress_parallel.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
        self.L = L

    def compress_parallel(self, data, with_sizes: bool = False):
        a = np.ascontiguousarray(np.frombuffer(bytes(data), np.uint8) if not isinstance(data, np.ndarray) else data,
                                 dtype=np.uint8)
        nb = (a.size + BLOCK - 1) // BLOCK
        out = np.empty(10 + a.size + nb * 1010 + 16, dtype=np.uint8)
        sizes = np.zeros(max(nb, 1), dtype=np.uint32)
        n = self.L.oracle_compress_parallel(a.ctypes.data, a.size, out.ctypes.data, sizes.ctypes.data)
        res = out[:n].copy()
        return (res, sizes[:nb]) if with_sizes else res

    # framegen.frame_compress_ref asks its "oracle" for compress(data, mode, with_sizes=True)
    def compress(self, data, mode: int = MODE_PARALLEL, with_sizes: bool = False):
        assert mode == MODE_PARALLEL
        return self.compress_parallel(data, with_sizes)


@pytest.fixture(scope="session")
def model(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("parallel_model") / "libparallel_parse.so")
    subprocess.run(["gcc", "-O2", "-shared", "-fPIC", "-Wall", "-Wextra", "-Werror",
                    "-I", os.path.join(ROOT, "lightweight-snappy_b200", "csrc"),
                    os.path.join(ROOT, "tests", "parallel_parse.c"), "-o", so], check=True)
    return ParallelModel(so)


# ---------------------------------------------------------------------------------------------- inputs
def _rand(seed: int, n: int) -> np.ndarray:
    return np.random.default_rng(seed).integers(0, 256, n, dtype=np.uint8)


def _text(n: int, first_segment: int = 0) -> np.ndarray:
    return corpus.make_corpus("text", n, first_segment=first_segment).numpy()


def _hash14(keys: np.ndarray) -> np.ndarray:
    return ((keys.astype(np.uint64) * 0x1E35A7BD) & 0xFFFFFFFF) >> 18


def _colliding_keys(count: int) -> list[bytes]:
    """Distinct 4-byte keys that all land in one table slot."""
    keys = np.random.default_rng(7).integers(0, 2**32, 1 << 20, dtype=np.uint64).astype(np.uint32)
    h = _hash14(keys)
    slot = np.bincount(h.astype(np.int64)).argmax()
    same = np.unique(keys[h == slot])[:count]
    assert same.size == count
    return [int(k).to_bytes(4, "little") for k in same]


def _far_match() -> np.ndarray:
    """The farthest copy a block can hold: the last 4 bytes repeat the first 4 (offset 65532).  Zeros in
    between, so that no other position shares the key's table slot."""
    a = np.zeros(BLOCK, np.uint8)
    a[:4] = a[BLOCK - 4:] = np.frombuffer(b"\x9a\xbc\xde\xf1", np.uint8)
    return a


def _tail_keys() -> np.ndarray:
    a = _rand(12, BLOCK + 100)
    a[BLOCK - 12:BLOCK] = np.frombuffer(b"wxyzwxyzwxyz", np.uint8)  # equal keys at the last positions of block 0
    a[-8:] = np.frombuffer(b"abcdabcd", np.uint8)                  # ... and of the short last block
    return a


def _collisions() -> np.ndarray:
    keys = _colliding_keys(8)
    rng = np.random.default_rng(13)
    return np.frombuffer(b"".join(keys[i] for i in rng.integers(0, 8, 40000)), np.uint8).copy()


def _max_records() -> np.ndarray:
    """Copies of exactly four bytes back to back: words drawn from a small vocabulary whose words share no
    byte, so no match runs on."""
    words = [bytes([4 * i + j for j in range(4)]) for i in range(64)]
    rng = np.random.default_rng(14)
    return np.frombuffer(b"".join(words[i] for i in rng.integers(0, 64, 3 * BLOCK // 4)), np.uint8).copy()


def _max_expansion() -> np.ndarray:
    """61 fresh bytes (a literal with a two-byte header) then 4 bytes repeated from 4 KiB back (a
    three-byte copy), over and over: the most stream bytes per input byte a parse can be made to write."""
    a = _rand(15, 2 * BLOCK)
    for p in range(4096 + 61, a.size - 4, 65):
        a[p:p + 4] = a[p - 4096:p - 4092]
    return a


def _skip_then_text() -> np.ndarray:
    """Random bytes, then text, then random again inside one block and in the next: the steps without a candidate
    are skipped (1, 2, 4, 8 steps) and the parse must pick the text up where the skipping lets it look again."""
    a = _rand(16, 2 * BLOCK + 5000)
    a[20000:50000] = _text(30000, 2)
    a[BLOCK + 9000:BLOCK + 13000] = _text(4000, 3)
    return a


def _periodic(period: int, n: int = 100000) -> np.ndarray:
    return np.resize(_rand(100 + period, period), n)


EDGE_SIZES = [0, 1, 3, 4, 5, 15, 16, 17, SLICE - 1, SLICE, SLICE + 1, BLOCK - 1, BLOCK, BLOCK + 1, BLOCK + 3]


def _inputs() -> dict[str, callable]:
    cases = {f"text_n{n}": (lambda n=n: _text(max(n, 1))[:n]) for n in EDGE_SIZES}
    cases.update({f"mixed_n{n}": (lambda n=n: corpus.make_corpus("mixed", max(n, 1), first_segment=2).numpy()[:n])
                  for n in (SLICE + 1, BLOCK + 3)})
    cases.update({
        "text_1mib": lambda: _text(1 << 20, 1),
        "mixed_3mib": lambda: corpus.make_corpus("mixed", (3 << 20) + 4321).numpy(),
        "zeros": lambda: np.zeros(3 * BLOCK + 77, np.uint8),
        "far_match": _far_match,
        "tail_keys": _tail_keys,
        "collisions": _collisions,
        "max_records": _max_records,
        "max_expansion": _max_expansion,
        "random": lambda: datasets.gen("corpus:random:7:0:200000"),
        "skip_then_text": _skip_then_text,
    })
    cases.update({f"period{k}": (lambda k=k: _periodic(k)) for k in range(1, 8)})
    return cases


INPUTS = _inputs()


# ---------------------------------------------------------------------------------------------- checks
def _elements(block: bytes):
    """(is_copy, length) of every element of one block's bytes (a valid block, as the model writes it)."""
    ip, out = 0, []
    while ip < len(block):
        tag = block[ip]
        if tag & 3 == 0:
            m = tag >> 2
            if m < 60:
                ip += 1
            else:
                k = m - 59
                m = int.from_bytes(block[ip + 1:ip + 1 + k], "little")
                ip += 1 + k
            out.append((False, m + 1))
            ip += m + 1
        else:
            out.append((True, 0))
            ip += (2, 3, 5)[(tag & 3) - 1]
    return out


def _check_stream(data: np.ndarray, stream: np.ndarray, sizes: np.ndarray, oracle):
    if data.size == 0:
        assert stream.size == 0, "an empty input gives an empty stream"
        return
    raw = stream.tobytes()
    got, reason = strict_ref.strict_decode(raw) if data.size <= (4 << 20) else (oracle.decompress(stream).tobytes(), "")
    assert got == data.tobytes(), f"strict decode: {reason}"
    assert np.array_equal(oracle.decompress(stream, data.size), data), "oracle decode"
    index, framed, largest = strict_ref.strict_layout(raw)
    assert index is not None and framed, "every element and every copy source stays inside its 64 KiB block"
    assert largest <= MAX_BLOCK_BYTES
    assert int(sizes.max()) <= MAX_BLOCK_BYTES
    pos = len(framegen.varint(data.size))
    assert index[0] == pos and len(index) == sizes.size + 1
    for b, s in enumerate(sizes):
        assert index[b + 1] - index[b] == s
        els = _elements(raw[pos:pos + int(s)])
        if not any(c for c, _ in els):
            n_b = min(BLOCK, data.size - b * BLOCK)
            assert els == [(False, n_b)], f"block {b} has no copy: it must be one literal"
        pos += int(s)


# ---------------------------------------------------------------------------------------------- CPU tests
@pytest.mark.parametrize("name", list(INPUTS))
def test_model_stream_invariants(model, oracle, name):
    data = INPUTS[name]()
    stream, sizes = model.compress_parallel(data, with_sizes=True)
    _check_stream(data, stream, sizes, oracle)
    assert np.array_equal(model.compress_parallel(data), stream), "deterministic"


def test_model_special_inputs_take_the_paths_they_are_for(model):
    recs = sum(c for c, _ in _elements(model.compress_parallel(_max_records()).tobytes()[3:]))
    assert recs > 10000, "max_records: most positions should start a 4-byte copy"
    exp = model.compress_parallel(_max_expansion())
    assert exp.size > _max_expansion().size, "max_expansion: the stream should be longer than the input"
    far = model.compress_parallel(_far_match()).tobytes()
    assert far.endswith(bytes([(4 - 1) << 2 | 2]) + (BLOCK - 4).to_bytes(2, "little")), "copy at offset 65532"


@pytest.mark.parametrize("kind,limit", [("text", 0.95), ("lowent", 1.05), ("random", 1.001), ("mixed", 1.00)])
def test_model_size_against_hash_mode(model, oracle, kind, limit):
    data = corpus.make_corpus(kind, 8 << 20).numpy()
    par, hsh = model.compress_parallel(data).size, oracle.compress(data, 0).size
    assert par / hsh <= limit, f"{kind}: {par} / {hsh} = {par / hsh:.4f} > {limit}"


# ---------------------------------------------------------------------------------------------- GPU tests
def _same(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    if got.size != want.size or not np.array_equal(got, want):
        m = min(got.size, want.size)
        i = int(np.argmax(got[:m] != want[:m])) if m and not np.array_equal(got[:m], want[:m]) else m
        raise AssertionError(f"{what}: sizes {got.size} vs {want.size}, first difference at byte {i} (block {i // BLOCK})")


def _compress_range(data: np.ndarray, mode: int, pieces: list[int]) -> np.ndarray:
    """snappy_b200_compress_host_range over consecutive ranges (whole blocks but the last), concatenated."""
    L, parts, lo = api.lib(), [], 0
    for k, hi in enumerate(pieces + [data.size]):
        a = np.ascontiguousarray(data[lo:hi])
        out = np.empty(api.max_compressed_bytes(a.size) + 16, np.uint8)
        n = C.c_uint64(0)
        rc = L.snappy_b200_compress_host_range(a.ctypes.data, a.size, mode, out.ctypes.data, out.size, C.byref(n), None,
                                               data.size if k == 0 else 0)
        assert rc == 0, api.lib().snappy_b200_last_error()
        parts.append(out[:n.value])
        lo = hi
    return np.concatenate(parts)


def _libc():
    libc = C.CDLL(None)
    libc.fopen.restype = C.c_void_p
    libc.fopen.argtypes = [C.c_char_p, C.c_char_p]
    libc.fclose.argtypes = [C.c_void_p]
    return libc


def _cli(*args, check=True):
    return subprocess.run([api.CLI_PATH, *map(str, args)], check=check, timeout=600, capture_output=True)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(INPUTS))
def test_device_and_host_match_the_model(model, name):
    import torch
    data = INPUTS[name]()
    want = model.compress_parallel(data)
    _same(api.compress_host(data, MODE_PARALLEL), want, "compress_host")
    stream, offs = api.compress_host_indexed(data, MODE_PARALLEL)
    _same(stream, want, "compress_host_indexed")
    if data.size:
        index, _, _ = strict_ref.strict_layout(want.tobytes())
        assert np.array_equal(offs, np.array(index, np.uint64)), "side index"
        codec = api.DeviceCodec(data.size)
        d = torch.from_numpy(data).cuda()
        codec.compress(d, MODE_PARALLEL)
        _same(codec.result_stream().cpu().numpy(), want, "compress_device")
        assert np.array_equal(codec.block_offsets.cpu().numpy().astype(np.uint64), offs), "device block offsets"
        codec.compress_framed(d, MODE_PARALLEL)
        _same(codec.result_stream().cpu().numpy(),
              np.frombuffer(framegen.frame_compress_ref(model, data, MODE_PARALLEL), np.uint8), "frame_compress_device")
        if data.size > 2 * BLOCK:
            _same(_compress_range(data, MODE_PARALLEL, [BLOCK, 2 * BLOCK]), want, "compress_host_range pieces")
    _same(np.frombuffer(api.compress_framed(data, MODE_PARALLEL).tobytes(), np.uint8),
          np.frombuffer(framegen.frame_compress_ref(model, data, MODE_PARALLEL), np.uint8), "frame_compress_host")


@pytest.mark.gpu
def test_large_mixed_every_entry_point(model, tmp_path):
    """256 MiB of mixed data: device, host (several pipeline chunks), ranges, multi-device, framed, and the
    command line -p, -p -i, -p -f, each equal to the model; the streams decode through every decoder."""
    import torch
    n = (256 << 20) + 12345
    data_t = corpus.make_corpus("mixed", n, device="cuda", first_segment=7).contiguous()
    data = data_t.cpu().numpy()
    want, sizes = model.compress_parallel(data, with_sizes=True)
    index = np.concatenate([[len(framegen.varint(n))], len(framegen.varint(n)) + np.cumsum(sizes)]).astype(np.uint64)

    codec = api.DeviceCodec(n)
    codec.compress(data_t, MODE_PARALLEL)
    _same(codec.result_stream().cpu().numpy(), want, "compress_device")
    # two calls and two CUDA streams at once give the same bytes
    other = api.DeviceCodec(n)
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    codec.compress(data_t, MODE_PARALLEL)
    with torch.cuda.stream(side):
        other.compress(data_t, MODE_PARALLEL)
    torch.cuda.synchronize()
    _same(codec.result_stream().cpu().numpy(), want, "second call")
    _same(other.result_stream().cpu().numpy(), want, "concurrent call on another stream")
    del other

    stream, offs = api.compress_host_indexed(data, MODE_PARALLEL)
    _same(stream, want, "compress_host_indexed")
    assert np.array_equal(offs, index)
    _same(_compress_range(data, MODE_PARALLEL, [64 << 20, (64 << 20) + BLOCK, 200 << 20]), want, "compress_host_range")
    n_dev = torch.cuda.device_count()
    _same(api.compress_host_multi(data, MODE_PARALLEL, 1), want, "compress_host_multi, 1 device")
    if n_dev >= 2:
        got, moffs = api.compress_host_multi(data, MODE_PARALLEL, 2, with_index=True)
        _same(got, want, "compress_host_multi, 2 devices")
        assert np.array_equal(moffs, index)
    framed_want = framegen.frame_compress_ref(model, data, MODE_PARALLEL)
    _same(np.frombuffer(api.compress_framed(data, MODE_PARALLEL).tobytes(), np.uint8),
          np.frombuffer(framed_want, np.uint8), "frame_compress_host")

    # decoders
    _same(api.decompress_host(want), data, "decompress_host")
    _same(api.decompress_host_indexed(want, offs), data, "decompress_host_indexed")
    _same(api.decompress_framed(np.frombuffer(framed_want, np.uint8)), data, "frame_decompress_host")
    s_t = torch.from_numpy(want).cuda()
    hdr = len(framegen.varint(n))
    out = torch.zeros(n, dtype=torch.uint8, device="cuda")
    codec.decompress(s_t, want.size, hdr, n, out)
    codec.check_status()
    assert torch.equal(out, data_t), "decompress_device"
    assert np.array_equal(codec.block_offsets.cpu().numpy().astype(np.uint64), index), "K0 block offsets"
    out.zero_()
    codec.decompress_async(s_t, want.size, hdr, n, out)
    codec.check_status()
    assert torch.equal(out, data_t), "decompress_device_async"
    out.zero_()
    codec.decompress_indexed(s_t, torch.from_numpy(offs.astype(np.int64)).cuda(), n, out)
    codec.check_status()
    assert torch.equal(out, data_t), "decompress_device_indexed with the compressor's offsets"
    del codec, out, s_t

    # command line and FILE* layer
    src = tmp_path / "in.bin"
    src.write_bytes(data.tobytes())
    _cli("-p", "-r", src, tmp_path / "p.snp")
    _same(np.fromfile(tmp_path / "p.snp", np.uint8), want, "snappy_b200 -p")
    _cli("-p", "-i", src, tmp_path / "pi.snp")
    _same(np.fromfile(tmp_path / "pi.snp", np.uint8), want, "snappy_b200 -p -i")
    idx = np.fromfile(str(tmp_path / "pi.snp") + ".idx", np.uint64)
    assert idx[1] == n and idx[2] == api.block_count(n) and np.array_equal(idx[3:], index)
    _cli("-p", "-f", src, tmp_path / "p.sz")
    assert (tmp_path / "p.sz").read_bytes() == framed_want, "snappy_b200 -p -f"
    for args, name in ((["-d"], "p.snp"), (["-d", "-i"], "pi.snp"), (["-f", "-d"], "p.sz")):
        back = tmp_path / (name + ".back")
        _cli(*args, tmp_path / name, back)
        assert back.read_bytes() == data.tobytes(), f"snappy_b200 {' '.join(args)}"
        back.unlink()
    # snappy_b200_decompress_file, called directly
    libc, L = _libc(), api.lib()
    fi, fo = libc.fopen(str(tmp_path / "p.snp").encode(), b"rb"), libc.fopen(str(tmp_path / "df.bin").encode(), b"wb")
    rc = L.snappy_b200_decompress_file(fi, fo)
    libc.fclose(fi), libc.fclose(fo)
    assert rc == 0 and (tmp_path / "df.bin").read_bytes() == data.tobytes(), "snappy_b200_decompress_file"


@pytest.mark.gpu
def test_file_calls_with_the_parallel_mode(model, tmp_path):
    """compress_file_indexed with index_out == NULL is the plain FILE* compressor; frame_compress_file."""
    data = corpus.make_corpus("mixed", (5 << 20) + 99, first_segment=4).numpy()
    src = tmp_path / "in.bin"
    src.write_bytes(data.tobytes())
    libc, L = _libc(), api.lib()
    for fn, out, want in (
            (lambda fi, fo: L.snappy_b200_compress_file_indexed(fi, data.size, MODE_PARALLEL, fo, None), "c.snp",
             model.compress_parallel(data).tobytes()),
            (lambda fi, fo: L.snappy_b200_frame_compress_file(fi, fo, MODE_PARALLEL), "c.sz",
             framegen.frame_compress_ref(model, data, MODE_PARALLEL))):
        fi, fo = libc.fopen(str(src).encode(), b"rb"), libc.fopen(str(tmp_path / out).encode(), b"wb")
        rc = fn(fi, fo)
        libc.fclose(fi), libc.fclose(fo)
        assert rc == 0, L.snappy_b200_last_error()
        assert (tmp_path / out).read_bytes() == want, out


@pytest.mark.gpu
def test_unknown_mode_is_an_argument_error(tmp_path):
    import torch
    L, bad = api.lib(), 3
    data = np.arange(100000, dtype=np.uint32).astype(np.uint8)
    out = np.empty(api.max_compressed_bytes(data.size) + 4096, np.uint8)
    offs = np.zeros(api.block_count(data.size) + 1, np.uint64)
    n = C.c_uint64(0)
    p, o = data.ctypes.data, out.ctypes.data
    codec = api.DeviceCodec(data.size)
    d = torch.from_numpy(data).cuda()
    src = tmp_path / "in.bin"
    src.write_bytes(data.tobytes())
    libc = _libc()
    before = api.launch_count()
    calls = {
        "compress_device": lambda: L.snappy_b200_compress_device(
            d.data_ptr(), data.size, bad, codec.stream_buf.data_ptr(), codec.comp_capacity, codec.out_bytes.data_ptr(),
            None, codec.status.data_ptr(), codec.workspace.data_ptr(), codec.workspace.numel(), None),
        "frame_compress_device": lambda: L.snappy_b200_frame_compress_device(
            d.data_ptr(), data.size, bad, codec.stream_buf.data_ptr(), codec.stream_buf.numel(),
            codec.out_bytes.data_ptr(), codec.status.data_ptr(), codec.workspace.data_ptr(), codec.workspace.numel(),
            None),
        "compress_host": lambda: L.snappy_b200_compress_host(p, data.size, bad, o, out.size, C.byref(n)),
        "compress_host_indexed": lambda: L.snappy_b200_compress_host_indexed(p, data.size, bad, o, out.size, C.byref(n),
                                                                             offs.ctypes.data),
        "compress_host_range": lambda: L.snappy_b200_compress_host_range(p, data.size, bad, o, out.size, C.byref(n),
                                                                         None, data.size),
        "compress_host_multi": lambda: L.snappy_b200_compress_host_multi(p, data.size, bad, o, out.size, C.byref(n),
                                                                         None, 2),
        "compress_host_multi_range": lambda: L.snappy_b200_compress_host_multi_range(
            p, data.size, bad, o, out.size, C.byref(n), None, 2, data.size),
        "frame_compress_host": lambda: L.snappy_b200_frame_compress_host(p, data.size, bad, o, out.size, C.byref(n)),
    }
    for name, call in calls.items():
        assert call() == api.ERR_ARG, name
    for name in ("frame_compress_file", "compress_file_indexed"):
        fi, fo = libc.fopen(str(src).encode(), b"rb"), libc.fopen(str(tmp_path / "o").encode(), b"wb")
        rc = (L.snappy_b200_frame_compress_file(fi, fo, bad) if name == "frame_compress_file"
              else L.snappy_b200_compress_file_indexed(fi, data.size, bad, fo, None))
        libc.fclose(fi), libc.fclose(fo)
        assert rc == api.ERR_ARG, name
    torch.cuda.synchronize()
    assert api.launch_count() == before, "nothing may be launched for an unknown mode"


@pytest.mark.gpu
def test_workspace_sized_for_hash_mode_is_too_small():
    import torch
    L, n = api.lib(), (3 << 20) + 5
    hash_ws = int(L.snappy_b200_compress_workspace_bytes(n, api.MODE_HASH))
    assert int(L.snappy_b200_compress_workspace_bytes(n, api.MODE_BST)) == hash_ws
    assert int(L.snappy_b200_compress_workspace_bytes(n, MODE_PARALLEL)) > hash_ws
    frame_ws = int(L.snappy_b200_frame_compress_workspace_bytes(n, api.MODE_HASH))
    assert int(L.snappy_b200_frame_compress_workspace_bytes(n, MODE_PARALLEL)) > frame_ws
    d = torch.zeros(n, dtype=torch.uint8, device="cuda")
    ws = torch.empty(max(hash_ws, frame_ws), dtype=torch.uint8, device="cuda")
    out = torch.empty(api.max_compressed_bytes(n) + 64, dtype=torch.uint8, device="cuda")
    small = torch.zeros(4, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    before = api.launch_count()
    assert L.snappy_b200_compress_device(d.data_ptr(), n, MODE_PARALLEL, out.data_ptr(), out.numel(), small.data_ptr(),
                                         None, small[2:].data_ptr(), ws.data_ptr(), hash_ws, None) == api.ERR_ARG
    assert L.snappy_b200_frame_compress_device(d.data_ptr(), n, MODE_PARALLEL, out.data_ptr(), out.numel(),
                                               small.data_ptr(), small[2:].data_ptr(), ws.data_ptr(), frame_ws,
                                               None) == api.ERR_ARG
    assert api.launch_count() == before
    # the same workspace is enough for hash mode
    assert L.snappy_b200_compress_device(d.data_ptr(), n, api.MODE_HASH, out.data_ptr(), out.numel(), small.data_ptr(),
                                         None, small[2:].data_ptr(), ws.data_ptr(), hash_ws, None) == 0
    torch.cuda.synchronize()
