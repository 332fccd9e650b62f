"""The Snappy framing format (include/snappy_b200.h, "framing format"): CRC-32C, the writer rule, the strict
unframer (tests/framegen.py) as the arbiter, and the library's framed calls against them.

CPU part: the reference CRC against RFC 3720 and a bitwise CRC, the golden streams, the arbiter on valid and mutated
streams, snappy_b200_frame_uncompressed_length (host only), and the framed compute calls failing without a device.
GPU part (-m gpu): byte-identical streams through every framed entry point, round trips, every foreign stream and
mutant with the arbiter's verdict, and a CUDA-graph capture of the enqueue-only device call."""
from __future__ import annotations

import hashlib
import os
import subprocess

import numpy as np
import pytest

import datasets
import framegen
from lightweight_snappy_b200 import api, corpus

# RFC 3720 B.4: input -> CRC-32C, and the masked CRC field of the one chunk that framing it gives
RFC = [(bytes(32), 0x8A9136AA, "faffd70f"), (b"\xff" * 32, 0x62A8AB43, "29b009f9"),
       (bytes(range(32)), 0x46DD794E, "92781f95"), (bytes(range(31, -1, -1)), 0x113FDB5C, "570d3b59")]
GOLDEN_123456789 = bytes.fromhex("ff060000734e61507059" "010d0000" "e5b08ac7" "313233343536373839")

SIZES = [0, 1, 65536, 65537]


@pytest.fixture(scope="module")
def L():
    if not os.path.exists(api.LIB_PATH):
        api.build()
    return api.lib()


def _have_gpu() -> bool:
    try:
        return api.device_count() > 0
    except Exception:
        return False


def _specs():
    specs = []
    for n in datasets.boundary_sizes():
        specs += [f"corpus:text:2:{n % 1000}:{n}", f"sym:5:{n}:{n}", f"lz:{n}:{n}", f"corpus:lowent:5:{n % 777}:{n}"]
    specs += [f"period:{p}:{p}:{n}" for p in (1, 2, 3, 5, 64, 65, 2047, 2048, 2049) for n in (4100, 66000)]
    specs += [f"corpus:random:7:0:{n}" for n in (1, 100, 65536, 65537, 140000)]
    specs += [f"sym:{k}:{k}:{70000}" for k in (1, 2, 4, 16, 64, 200)]
    return specs


# ---------------------------------------------------------------------------------------------- CPU
def test_crc32c_vectors():
    assert framegen.crc32c(b"123456789") == 0xE3069283
    assert framegen.masked_crc(b"123456789") == 0xC78AB0E5
    for data, crc, field in RFC:
        assert framegen.crc32c(data) == crc
        assert framegen.crc32c_bitwise(data) == crc
        assert framegen.masked_crc(data).to_bytes(4, "little").hex() == field
    rng = np.random.default_rng(5)
    for n in (0, 1, 7, 255, 4097):
        b = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        assert framegen.crc32c(b) == framegen.crc32c_bitwise(b)
    big = rng.integers(0, 256, 3 * 65536 + 77, dtype=np.uint8)
    assert framegen.block_crcs(big) == [framegen.crc32c(big[i:i + 65536].tobytes()) for i in range(0, big.size, 65536)]
    assert framegen.mask(0) == 0xA282EAD8


def test_reference_writer_golden(oracle):
    assert framegen.frame_compress_ref(oracle, np.frombuffer(b"123456789", np.uint8)) == GOLDEN_123456789
    assert framegen.frame_compress_ref(oracle, np.zeros(0, np.uint8)) == framegen.STREAM_ID
    for data, _, field in RFC:
        s = framegen.frame_compress_ref(oracle, np.frombuffer(data, np.uint8))
        assert s[14:18].hex() == field


def test_arbiter_agrees_with_writer(oracle):
    for spec in _specs()[::3] + ["corpus:text:1:0:300000"]:
        data = datasets.gen(spec)
        for mode in (0, 1):
            s = framegen.frame_compress_ref(oracle, data, mode)
            assert len(s) <= 10 + data.size + 8 * -(-data.size // 65536)
            out, verdict = framegen.unframe(s)
            assert verdict == "ok" and out == data.tobytes(), spec


def test_arbiter_on_foreign_streams_and_mutants(oracle):
    for name, s, data in framegen.foreign_streams(oracle):
        assert framegen.unframe(s) == (data, "ok"), name
        assert framegen.total_length(s) == len(data), name
    s = framegen.frame_compress_ref(oracle, datasets.gen("corpus:text:2:0:200000"))
    verdicts = dict((name, framegen.unframe(m)[1]) for name, m in framegen.mutants(s))
    assert verdicts["no-identifier"] == verdicts["unskippable-0x02"] == verdicts["n>65536"] == "corrupt"
    assert verdicts["uncompressed>65536"] == verdicts["truncated-payload"] == verdicts["length-past-end"] == "corrupt"
    assert all(v == "checksum" for k, v in verdicts.items() if k.startswith("crc-flip"))
    assert all(v != "ok" for v in verdicts.values())
    # a flipped data byte of an uncompressed chunk is well formed: only the checksum can catch it
    u = framegen.STREAM_ID + framegen.data_chunk(b"abcdefgh")
    assert framegen.unframe(u[:-1] + b"i") == (None, "checksum")


def test_frame_uncompressed_length_without_device(L, oracle):
    """Host only: exact lengths on valid streams, ERR_CORRUPT on header mutants."""
    for name, s, data in framegen.foreign_streams(oracle):
        assert api.framed_uncompressed_length(np.frombuffer(s, np.uint8)) == len(data), name
    for n in SIZES:
        s = framegen.frame_compress_ref(oracle, datasets.gen(f"corpus:random:7:0:{n}") if n else np.zeros(0, np.uint8))
        assert api.framed_uncompressed_length(np.frombuffer(s, np.uint8)) == n
    assert api.framed_uncompressed_length(np.zeros(0, np.uint8)) == 0
    s = framegen.frame_compress_ref(oracle, datasets.gen("corpus:text:2:0:200000"))
    for name, m in framegen.mutants(s):
        want = framegen.total_length(m)
        if want is None:
            with pytest.raises(api.SnappyError) as e:
                api.framed_uncompressed_length(np.frombuffer(m, np.uint8))
            assert e.value.code == api.ERR_CORRUPT, name
            assert "offset" in str(e.value), name
        else:
            assert api.framed_uncompressed_length(np.frombuffer(m, np.uint8)) == want, name


def test_framed_calls_fail_without_device(L):
    if _have_gpu():
        pytest.skip("a device is present")
    for call in (lambda: api.compress_framed(b"abc"), lambda: api.compress_framed(b""),
                 lambda: api.decompress_framed(GOLDEN_123456789), lambda: api.decompress_framed(framegen.STREAM_ID)):
        with pytest.raises(api.SnappyError):
            call()


# ---------------------------------------------------------------------------------------------- GPU
def _check_framed(oracle, data, mode, what):
    want = framegen.frame_compress_ref(oracle, data, mode)
    got = api.compress_framed(data, mode).tobytes()
    assert got == want, f"{what} mode {mode}: framed stream differs from the reference writer"
    back = api.decompress_framed(np.frombuffer(got, np.uint8))
    assert np.array_equal(back[:data.size], data) and back.size == data.size, f"{what} mode {mode}: round trip"


@pytest.mark.gpu
def test_golden_streams():
    assert api.compress_framed(b"123456789").tobytes() == GOLDEN_123456789
    assert api.compress_framed(b"", api.MODE_BST).tobytes() == framegen.STREAM_ID
    for data, _, field in RFC:
        for mode in (0, 1):
            s = api.compress_framed(data, mode).tobytes()
            assert s[14:18].hex() == field
            assert api.decompress_framed(s).tobytes() == data
    assert api.decompress_framed(GOLDEN_123456789).tobytes() == b"123456789"
    assert api.decompress_framed(b"").size == 0
    assert api.decompress_framed(framegen.STREAM_ID).size == 0


@pytest.mark.gpu
def test_framed_against_reference_writer(oracle):
    for spec in _specs():
        data = datasets.gen(spec)
        for mode in (0, 1):
            _check_framed(oracle, data, mode, spec)
    for n in SIZES:
        for kind in ("text", "random"):
            data = datasets.gen(f"corpus:{kind}:3:0:{n}") if n else np.zeros(0, np.uint8)
            for mode in (0, 1):
                _check_framed(oracle, data, mode, f"{kind} {n}")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["mixed", "text", "lowent", "random"])
def test_framed_64mib_corpora(oracle, kind):
    import torch
    n = 64 << 20
    data = corpus.make_corpus(kind, n, device="cuda")
    host = data.cpu().numpy()
    codec = api.DeviceCodec(n)
    for mode in (0, 1):
        # the BST oracle is slow on text: 16 MiB of it, as in test_gpu_parity
        h, d = (host[: 16 << 20], data[: 16 << 20]) if mode == 1 and kind in ("text", "mixed") else (host, data)
        want = framegen.frame_compress_ref(oracle, h, mode)
        got = api.compress_framed(h, mode).tobytes()
        assert got == want, f"{kind} mode {mode}: host API"
        codec.compress_framed(d, mode)
        dev = codec.result_stream().cpu().numpy().tobytes()
        assert dev == want, f"{kind} mode {mode}: device API"
        back = api.decompress_framed(np.frombuffer(got, np.uint8))
        assert np.array_equal(back, h), f"{kind} mode {mode}: round trip"
    del data, codec
    torch.cuda.empty_cache()


def _shard_worker(args):
    shard, shard_bytes = args
    import oracle_lib
    from lightweight_snappy_b200 import corpus as cp
    data = cp.make_corpus("mixed", shard_bytes, first_segment=shard * (shard_bytes >> 20)).numpy()
    s = framegen.frame_compress_ref(oracle_lib.Oracle(), data, 0, identifier=False)
    return len(s), hashlib.sha256(s).hexdigest(), hashlib.sha256(data.tobytes()).hexdigest()


@pytest.mark.gpu
def test_framed_256mib_mixed_by_shards(oracle):
    """256 MiB mixed, hash mode, compared with the reference writer shard by shard (SHA-256): chunks are
    independent, so the stream is the identifier followed by the framings of the 64 MiB shards."""
    import multiprocessing as mp
    shard, n = 64 << 20, 256 << 20
    data = corpus.make_corpus("mixed", n)
    host = data.numpy()
    got = api.compress_framed(host, 0)
    assert got[:10].tobytes() == framegen.STREAM_ID
    with mp.get_context("spawn").Pool(4) as pool:
        shards = pool.map(_shard_worker, [(s, shard) for s in range(n // shard)])
    off = 10
    for s, (ln, sha, data_sha) in enumerate(shards):
        assert hashlib.sha256(host[s * shard:(s + 1) * shard].tobytes()).hexdigest() == data_sha, f"corpus shard {s}"
        assert hashlib.sha256(got[off:off + ln].tobytes()).hexdigest() == sha, f"shard {s} differs"
        off += ln
    assert off == got.size
    back = api.decompress_framed(got)
    assert np.array_equal(back, host)


@pytest.mark.gpu
def test_foreign_streams_and_mutants(oracle):
    """Every valid foreign stream decodes exactly; every mutant gets the arbiter's verdict; a valid stream still
    decodes after each rejection."""
    code = {"corrupt": api.ERR_CORRUPT, "checksum": api.ERR_CHECKSUM}
    valid = framegen.frame_compress_ref(oracle, datasets.gen("corpus:text:2:0:200000"))
    valid_data = datasets.gen("corpus:text:2:0:200000")
    for name, s, data in framegen.foreign_streams(oracle):
        assert api.decompress_framed(np.frombuffer(s, np.uint8)).tobytes() == data, name
    cases = [(f"writer:{n}", m) for n, m in framegen.mutants(valid)]
    for name, s, _ in framegen.foreign_streams(oracle)[::3]:
        if framegen.walk(s)[0]:
            cases += [(f"{name}:{n}", m) for n, m in framegen.mutants(s)]
    for name, m in cases:
        out, verdict = framegen.unframe(m)
        if verdict == "ok":
            assert api.decompress_framed(np.frombuffer(m, np.uint8)).tobytes() == out, name
            continue
        with pytest.raises(api.SnappyError) as e:
            api.decompress_framed(np.frombuffer(m, np.uint8))
        assert e.value.code == code[verdict], f"{name}: {e.value} (want {verdict})"
        assert np.array_equal(api.decompress_framed(np.frombuffer(valid, np.uint8)), valid_data), f"after {name}"


@pytest.mark.gpu
def test_frame_device_api_cuda_graph(oracle):
    """The framed device call only enqueues: captured into a CUDA graph and replayed on new data."""
    import torch
    n = 24 << 20
    codec = api.DeviceCodec(n)
    data = corpus.make_corpus("mixed", n, device="cuda", first_segment=3).clone()
    codec.compress_framed(data, 0)
    want = framegen.frame_compress_ref(oracle, data.cpu().numpy(), 0)
    assert codec.result_stream().cpu().numpy().tobytes() == want
    side = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        side.synchronize()
        with torch.cuda.graph(g, stream=side):
            codec.compress_framed(data, 0)
    data.copy_(corpus.make_corpus("text", n, device="cuda"))
    want2 = framegen.frame_compress_ref(oracle, data.cpu().numpy(), 0)
    for _ in range(2):
        codec.stream_buf.zero_()
        codec.status.fill_(7)
        g.replay()
        torch.cuda.synchronize()
        assert int(codec.status.item()) == 0, "the captured memset and kernels leave a clean status"
        assert codec.result_stream().cpu().numpy().tobytes() == want2, "replayed stream"
    # empty input: the identifier alone, also on the device
    codec.compress_framed(torch.empty(0, dtype=torch.uint8, device="cuda"), 1)
    assert codec.result_stream().cpu().numpy().tobytes() == framegen.STREAM_ID


# ---------------------------------------------------------------------------------------------- FILE* / `-f`
def _cli(*args, env=None, stdin=None):
    return subprocess.run([api.CLI_PATH, *args], env={**os.environ, **(env or {})}, stdin=stdin,
                          capture_output=True)


def test_cli_f_with_i_is_a_usage_error(L, tmp_path):
    src = tmp_path / "in"
    src.write_bytes(b"abc")
    for flag in ("-c", "-b", "-d"):
        r = _cli("-f", "-i", flag, str(src), str(tmp_path / "out"))
        assert r.returncode != 0 and b"cannot be combined" in r.stderr


@pytest.mark.gpu
def test_cli_framed_against_reference_writer(oracle, tmp_path):
    """snappy_b200 -f -c / -b: byte-identical to the reference writer, also when the file is read in many chunks
    (SNAPPY_B200_FILE_CHUNK_MIB=1); -f -d gives the bytes back."""
    cases = [("empty", np.zeros(0, np.uint8)), ("one", datasets.gen("hex:41")),
             ("65537", datasets.gen("corpus:text:3:0:65537")), ("5mib", corpus.make_corpus("mixed", 5 << 20).numpy())]
    for name, data in cases:
        src, sz, back = tmp_path / f"{name}.bin", tmp_path / f"{name}.sz", tmp_path / f"{name}.back"
        src.write_bytes(data.tobytes())
        for flag, mode in (("-c", 0), ("-b", 1)):
            for env in ({}, {"SNAPPY_B200_FILE_CHUNK_MIB": "1"}):
                r = _cli("-f", flag, str(src), str(sz), env=env)
                assert r.returncode == 0, r.stderr
                assert sz.read_bytes() == framegen.frame_compress_ref(oracle, data, mode), f"{name} {flag} {env}"
            r = _cli("-f", "-d", str(sz), str(back))
            assert r.returncode == 0, r.stderr
            assert back.read_bytes() == data.tobytes(), f"{name} {flag}: -f -d"


@pytest.mark.gpu
def test_cli_framed_decompress_from_pipe(oracle, tmp_path):
    """-f -d reads a non-seekable input in 32 MiB windows and carries the incomplete chunk across: a 96 MiB stream
    of mixed corpus (several windows, chunks cut at window ends) and a foreign stream come back exactly; a
    mis-checksummed stream fails."""
    data = corpus.make_corpus("mixed", 96 << 20).numpy()
    sz, back = tmp_path / "big.sz", tmp_path / "big.back"
    sz.write_bytes(api.compress_framed(data, 0).tobytes())
    with open(sz, "rb") as f:
        p = subprocess.Popen(["cat"], stdin=f, stdout=subprocess.PIPE)
        r = _cli("-f", "-d", "/dev/stdin", str(back), stdin=p.stdout)
        p.stdout.close()
        p.wait()
    assert r.returncode == 0, r.stderr
    assert hashlib.sha256(back.read_bytes()).digest() == hashlib.sha256(data.tobytes()).digest()
    for name, s, want in framegen.foreign_streams(oracle)[::4]:
        r = subprocess.run(f"cat | {api.CLI_PATH} -f -d /dev/stdin {back}", shell=True, input=s, capture_output=True)
        assert r.returncode == 0, (name, r.stderr)
        assert back.read_bytes() == want, name
    u = framegen.STREAM_ID + framegen.data_chunk(b"abcdefgh")
    r = subprocess.run(f"cat | {api.CLI_PATH} -f -d /dev/stdin {back}", shell=True, input=u[:-1] + b"i",
                       capture_output=True)
    assert r.returncode != 0 and b"CRC-32C" in r.stderr
