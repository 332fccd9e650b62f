"""GPU parity tests (run on the B200 box with `-m gpu`): the CUDA path, called through the
C-ABI, against the CPU oracle and the golden vectors captured from the reference."""
import hashlib
import json
import os

import numpy as np
import pytest

import datasets
from lightweight_snappy_b200 import api, corpus

pytestmark = pytest.mark.gpu

GOLDEN = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden.json")))


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _first_diff(a, b):
    n = min(a.size, b.size)
    d = np.nonzero(a[:n] != b[:n])[0]
    return int(d[0]) if d.size else n


def _assert_same(got, want, what):
    if got.size != want.size or not np.array_equal(got, want):
        i = _first_diff(got, want)
        raise AssertionError(f"{what}: sizes {got.size} vs {want.size}, first difference at byte {i} "
                             f"(block {i // 65536}): got {got[i:i + 16].tobytes().hex()} want {want[i:i + 16].tobytes().hex()}")


@pytest.mark.parametrize("case", GOLDEN["cases"], ids=lambda c: c["spec"])
def test_golden_vectors(case):
    data = datasets.gen(case["spec"])
    assert _sha(data) == case["input_sha256"]
    for name, fn in (("hash", api.snappy_compress), ("bst", api.snappy_compress_bst)):
        s = fn(data)
        assert s.size == case[name]["len"], (name, s.size, case[name]["len"])
        assert _sha(s) == case[name]["sha256"], name
        _assert_same(api.snappy_decompress(s), data, f"roundtrip {name}")


def _fuzz_specs():
    specs = []
    for n in datasets.boundary_sizes():
        specs += [f"corpus:text:2:{n % 1000}:{n}", f"sym:5:{n}:{n}", f"lz:{n}:{n}", f"corpus:lowent:5:{n % 777}:{n}"]
    specs += [f"period:{p}:{p}:{n}" for p in (1, 2, 3, 5, 64, 65, 2047, 2048, 2049) for n in (4100, 66000)]
    specs += [f"corpus:random:7:0:{n}" for n in (1, 100, 65536, 65537, 140000)]
    specs += [f"sym:{k}:{k}:{70000}" for k in (1, 2, 4, 16, 64, 200)]
    return specs


def test_fuzz_against_oracle(oracle):
    for spec in _fuzz_specs():
        data = datasets.gen(spec)
        for mode, fn in ((0, api.snappy_compress), (1, api.snappy_compress_bst)):
            want = oracle.compress(data, mode)
            _assert_same(fn(data), want, f"{spec} mode {mode}")
        _assert_same(api.snappy_decompress(oracle.compress(data, 0)), data, f"{spec} decode(hash stream)")
        _assert_same(api.snappy_decompress(oracle.compress(data, 1)), data, f"{spec} decode(bst stream)")


def test_empty_input():
    assert api.snappy_compress(np.zeros(0, np.uint8)).size == 0
    assert api.snappy_compress_bst(np.zeros(0, np.uint8)).size == 0
    assert api.snappy_decompress(np.zeros(0, np.uint8)).size == 0


@pytest.mark.parametrize("kind", ["mixed", "text", "lowent", "random", "lowent_random"])
def test_device_api_64mib_against_oracle(oracle, kind):
    import torch
    n = 64 << 20 if kind in ("mixed", "lowent_random") else 16 << 20
    data = corpus.make_corpus(kind, n, device="cuda")
    host = data.cpu().numpy()
    codec = api.DeviceCodec(n)
    for mode in (0, 1):
        if mode == 1 and kind in ("text", "mixed") and n > (16 << 20):
            host_m, data_m = host[: 16 << 20], data[: 16 << 20]  # the BST oracle is slow on text
        else:
            host_m, data_m = host, data
        want, sizes = oracle.compress(host_m, mode, with_sizes=True)
        codec.compress(data_m, mode)
        got = codec.result_stream().cpu().numpy()
        _assert_same(got, want, f"{kind} mode {mode} stream")
        nb = api.block_count(host_m.size)
        offs = codec.block_offsets[: nb + 1].cpu().numpy()
        assert np.array_equal(np.diff(offs).astype(np.uint32), sizes), "side index"
        # decode with the side index ...
        out = torch.empty(host_m.size, dtype=torch.uint8, device="cuda")
        codec.decompress_indexed(codec.stream_buf, codec.block_offsets, host_m.size, out)
        codec.check_status()
        assert torch.equal(out, data_m)
        # ... and with the index rebuilt from the bare stream (K0)
        hdr = len(oracle.varint_encode(host_m.size))
        offs2 = torch.zeros(nb + 1, dtype=torch.int64, device="cuda")
        codec.index(codec.stream_buf, got.size, hdr, host_m.size, offs2)
        codec.check_status()
        assert np.array_equal(offs2.cpu().numpy(), offs), "K0 block offsets"
        assert api.index_rounds() <= 64, f"K0 needed {api.index_rounds()} relaxation rounds"
        want_offs, _ = oracle.block_index(want)
        assert np.array_equal(offs.astype(np.uint64), want_offs)
        # ... and the whole index-less path: K0 + segment-driven decoder
        out2 = torch.zeros(host_m.size, dtype=torch.uint8, device="cuda")
        offs3 = torch.zeros(nb + 1, dtype=torch.int64, device="cuda")
        codec.decompress(codec.stream_buf, got.size, hdr, host_m.size, out2, offs3)
        codec.check_status()
        assert torch.equal(out2, data_m), "index-less decode"
        assert np.array_equal(offs3.cpu().numpy(), offs)


def test_decoder_foreign_and_malformed_streams(oracle):
    # copy-4 elements (src/snappy_decompression.c:323-327) never come out of the compressors
    stream = b"\x08" + b"\x0cabcd" + bytes([(3 << 2) | 3, 4, 0, 0, 0])
    assert api.snappy_decompress(np.frombuffer(stream, np.uint8)).tobytes() == b"abcdabcd"
    # slide example: literal of 67 then copy-1 len 6 offset 63
    lit = bytes(range(67))
    stream = b"\x49" + b"\xf0\x42" + lit + b"\x09\x3f"
    assert api.snappy_decompress(np.frombuffer(stream, np.uint8)).tobytes() == lit + lit[4:10]
    for bad in (b"\x08\x0cabcd" + bytes([(3 << 2) | 2, 9, 0]),   # offset beyond the output
                b"\x08\x0cab",                                    # truncated literal
                b"\x04\x0cabcd\x0cabcd",                          # more output than declared
                b"\x20\x0cabcd"):                                 # less output than declared
        with pytest.raises(api.SnappyError):
            api.snappy_decompress(np.frombuffer(bad, np.uint8))


def test_decode_google_snappy_streams():
    pa = pytest.importorskip("pyarrow")
    codec = pa.Codec("snappy")
    for spec in ("corpus:text:0:0:300000", "corpus:lowent:1:0:200000", "corpus:random:2:0:70000", "rep:0:200000",
                 "lz:9:150000"):
        data = datasets.gen(spec)
        foreign = np.frombuffer(codec.compress(data.tobytes()).to_pybytes(), np.uint8)
        _assert_same(api.snappy_decompress(foreign), data, f"google stream of {spec}")
        # and Google's decoder accepts ours
        mine = api.snappy_compress(data)
        back = codec.decompress(mine.tobytes(), decompressed_size=data.size).to_pybytes()
        assert back == data.tobytes()


def test_roundtrip_properties_at_scale():
    """Size-independent properties at a size the oracle is too slow for: round trip,
    determinism, and block independence (a block's bytes do not depend on its neighbours)."""
    import torch
    n = 256 << 20
    data = corpus.make_corpus("mixed", n, device="cuda")
    codec = api.DeviceCodec(n)
    codec.compress(data, 0)
    s1 = codec.result_stream().clone()
    offs1 = codec.block_offsets.clone()
    out = torch.empty(n, dtype=torch.uint8, device="cuda")
    codec.decompress_indexed(s1, offs1, n, out)
    codec.check_status()
    assert torch.equal(out, data)
    codec.compress(data, 0)
    assert torch.equal(codec.result_stream(), s1), "compression is deterministic"
    # block independence: compress the second half alone, compare block bodies
    half = n // 2
    codec.compress(data[half:], 0)
    s2 = codec.result_stream().clone()
    offs2 = codec.block_offsets[: half // 65536 + 1].clone()
    b1 = s1[int(offs1[half // 65536]):]
    b2 = s2[int(offs2[0]):]
    assert torch.equal(b1, b2)
    ratio = n / s1.numel()
    assert 1.5 < ratio < 4.0, ratio
    # and against the oracle: 32 blocks spread over the 256 MiB, byte for byte
    import oracle_lib
    orc = oracle_lib.Oracle()
    offs = offs1.cpu().numpy()
    for b in np.linspace(0, n // 65536 - 1, 32).astype(np.int64):
        blk = data[b * 65536:(b + 1) * 65536].cpu().numpy()
        ref = orc.compress(blk, 0)
        vl = len(orc.varint_encode(blk.size))
        got = s1[int(offs[b]):int(offs[b + 1])].cpu().numpy()
        _assert_same(got, ref[vl:], f"block {b} vs oracle")


def test_host_pipeline_many_chunks(monkeypatch, oracle):
    """The chunked host pipeline (13 compress chunks, ~15 upload pieces, a ragged tail) gives the
    ORACLE's stream (and so does one device-resident call), from pageable and from page-locked buffers."""
    import torch
    monkeypatch.setenv("SNAPPY_B200_CHUNK_MIB", "16")   # 13 compress chunks, 4 in flight
    monkeypatch.setenv("SNAPPY_B200_PIECE_MIB", "8")    # ~15 upload pieces
    n = (200 << 20) + 12345
    data = corpus.make_corpus("mixed", n, device="cuda", first_segment=7)
    codec = api.DeviceCodec(n)
    codec.compress(data, 0)
    host = data.cpu()
    want = oracle.compress(host.numpy(), 0)
    _assert_same(codec.result_stream().cpu().numpy(), want, "device-resident stream vs oracle")
    _assert_same(oracle.decompress(want), host.numpy(), "oracle decoder on the stream")
    pinned = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    pinned.copy_(host)
    for src in (host.numpy(), pinned.numpy()):
        got = api.compress_host(src, api.MODE_HASH)
        _assert_same(got, want, "host pipeline stream")
    back = api.decompress_host(want)
    _assert_same(back, host.numpy(), "host pipeline decode")
    out_pinned = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    back2 = api.decompress_host(want, out=out_pinned.numpy())
    assert back2.size == n and torch.equal(out_pinned, host)
    # a stream cut short must be rejected, not mis-decoded
    with pytest.raises(api.SnappyError):
        api.decompress_host(want[: want.size - 70000])


def test_cli_roundtrip(tmp_path, oracle):
    import subprocess
    data = datasets.gen("corpus:mixed:0:900000:400000")
    src, snp, bsn, dec = (tmp_path / x for x in ("in.bin", "out.snp", "out.bsnp", "out.dec"))
    src.write_bytes(data.tobytes())
    subprocess.run([api.CLI_PATH, "-c", str(src), str(snp)], check=True)
    subprocess.run([api.CLI_PATH, "-b", "-r", str(src), str(bsn)], check=True)
    subprocess.run([api.CLI_PATH, "-d", str(snp), str(dec)], check=True)
    assert snp.read_bytes() == oracle.compress(data, 0).tobytes()
    assert bsn.read_bytes() == oracle.compress(data, 1).tobytes()
    assert dec.read_bytes() == data.tobytes()


def test_config0_reference_cli_64mib_text(tmp_path):
    """BASELINE.json configs[0]: the reference's own command line (oracle/_ref/snappy_ref, built
    unmodified from /root/reference/src) against ours on a 64 MiB text-like file: `-c` streams
    must be byte-identical, each decoder must invert the other's stream."""
    import subprocess
    import oracle_lib
    if not os.path.exists(oracle_lib.REF_BIN):
        pytest.skip("oracle/_ref/snappy_ref not built")
    data = corpus.make_corpus("text", 64 << 20, device="cuda").cpu().numpy()
    src = tmp_path / "text64.bin"
    src.write_bytes(data.tobytes())
    ours, theirs = tmp_path / "ours.snp", tmp_path / "ref.snp"
    subprocess.run([api.CLI_PATH, "-c", str(src), str(ours)], check=True)
    subprocess.run([oracle_lib.REF_BIN, "-c", str(src), str(theirs)], check=True)
    a, b = np.fromfile(ours, np.uint8), np.fromfile(theirs, np.uint8)
    _assert_same(a, b, "CLI -c stream vs reference CLI")
    # our decoder on the reference's stream, the reference's decoder on ours
    subprocess.run([api.CLI_PATH, "-d", str(theirs), str(tmp_path / "ours.dec")], check=True)
    _assert_same(np.fromfile(tmp_path / "ours.dec", np.uint8), data, "our -d on the reference stream")
    subprocess.run([oracle_lib.REF_BIN, "-d", str(ours), str(tmp_path / "ref.dec")], check=True)
    _assert_same(np.fromfile(tmp_path / "ref.dec", np.uint8), data, "reference -d on our stream")
    # BST path: same size (and in fact the same bytes) as the reference's -b
    subprocess.run([api.CLI_PATH, "-b", str(src), str(tmp_path / "ours.bsnp")], check=True)
    small = tmp_path / "text8.bin"
    small.write_bytes(data[: 8 << 20].tobytes())
    subprocess.run([api.CLI_PATH, "-b", str(small), str(tmp_path / "ours8.bsnp")], check=True)
    subprocess.run([oracle_lib.REF_BIN, "-b", str(small), str(tmp_path / "ref8.bsnp")], check=True)
    _assert_same(np.fromfile(tmp_path / "ours8.bsnp", np.uint8), np.fromfile(tmp_path / "ref8.bsnp", np.uint8),
                 "CLI -b stream vs reference CLI")


def test_decoders_on_random_valid_streams(oracle):
    """Element kinds and encodings the compressors never emit (tests/streamgen.py): both decoders
    and K0 against the oracle decoder."""
    import torch
    import streamgen
    cases = [(s, n, st) for s, (n, st) in enumerate([
        (1, "mixed"), (100, "mixed"), (4095, "copies"), (65536, "mixed"), (65537, "copies"), (70000, "bigliteral"),
        (200000, "copies"), (300001, "bigliteral"), (1 << 20, "mixed"), (3 << 20, "copies"), (5 << 20, "bigliteral")])]
    for seed, total, style in cases:
        stream, want = streamgen.make_stream(1000 + seed, total, style)
        assert np.array_equal(oracle.decompress(stream), want)
        # host API: K0 + segment-driven decoder
        _assert_same(api.snappy_decompress(stream), want, f"seg decoder {seed} {total} {style}")
        # window decoder with the oracle's block index
        offs, _ = oracle.block_index(stream)
        d_stream = torch.from_numpy(np.concatenate([stream, np.zeros(64, np.uint8)])).cuda()
        d_offs = torch.from_numpy(offs.astype(np.int64)).cuda()
        out = torch.zeros(total, dtype=torch.uint8, device="cuda")
        codec = api.DeviceCodec(max(total, 1 << 16))
        codec.decompress_indexed(d_stream, d_offs, total, out)
        codec.check_status()
        _assert_same(out.cpu().numpy(), want, f"window decoder {seed} {total} {style}")
        # K0 block offsets
        hdr = stream.size - (offs[-1] - offs[0]) if False else int(offs[0])
        got_offs = torch.zeros(len(offs), dtype=torch.int64, device="cuda")
        codec.index(d_stream, stream.size, hdr, total, got_offs)
        codec.check_status()
        assert np.array_equal(got_offs.cpu().numpy().astype(np.uint64), offs), f"K0 offsets {seed}"


@pytest.mark.gpu
def test_batch_tool_config4_small():
    """BASELINE configs[4] at reduced size: tools/batch64.py (block-range sharding, sub-batches,
    1 % oracle spot check, checksum) on a 256 MiB batch."""
    import json
    import subprocess
    import sys
    root = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "batch64.py"), "--gib", "0.25", "--sub-gib", "0.125"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert d["roundtrip_ok"] and d["checksum_ok"] and d["oracle_checked_fraction"] >= 0.01
    assert abs(d["ratio"] - 1.72) < 0.02


@pytest.mark.gpu
def test_selftest_driver():
    """SURVEY 8f-3: the snappy_test-shaped round-trip driver over generated fixtures (the six
    named files + 13 sizes x 5), both compressors, through the FILE*-based drop-in API."""
    import subprocess
    exe = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "lightweight-snappy_b200", "snappy_b200_test")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-1000:])
    assert "142 round trips, 0 failed" in r.stdout


@pytest.mark.gpu
def test_side_index_host_api(oracle, monkeypatch):
    """SURVEY 8f-4: the optional side index.  The stream is unchanged, the index equals the
    oracle's block index, the indexed decoder (no K0) inverts it, and a wrong index is reported."""
    monkeypatch.setenv("SNAPPY_B200_CHUNK_MIB", "4")   # several compress chunks
    monkeypatch.setenv("SNAPPY_B200_PIECE_MIB", "8")   # several decode pieces
    for spec in ("corpus:mixed:0:0:20000000", "corpus:text:1:100:65536", "corpus:lowent:2:0:65537", "hex:616263",
                 "corpus:random:5:0:1000000"):
        data = datasets.gen(spec)
        for mode in (0, 1):
            want = oracle.compress(data, mode)
            stream, offs = api.compress_host_indexed(data, mode)
            _assert_same(stream, want, f"{spec} mode {mode}: stream with index")
            ref_idx, _ = oracle.block_index(want)
            assert offs.tolist() == [int(x) for x in ref_idx], f"{spec} mode {mode}: index"
            _assert_same(api.decompress_host_indexed(stream, offs), data, f"{spec} mode {mode}: indexed decode")
    data = datasets.gen("corpus:mixed:0:0:400000")
    stream, offs = api.compress_host_indexed(data, 0)
    bad = offs.copy()
    bad[3] += 1
    with pytest.raises(api.SnappyError):
        api.decompress_host_indexed(stream, bad)
    bad = offs.copy()
    bad[2], bad[3] = offs[3], offs[2]
    with pytest.raises(api.SnappyError):
        api.decompress_host_indexed(stream, bad)


@pytest.mark.gpu
def test_cli_side_index(tmp_path):
    data = datasets.gen("corpus:mixed:0:0:5000000")
    src, comp, back, plain = tmp_path / "in", tmp_path / "c.snp", tmp_path / "back", tmp_path / "plain.snp"
    src.write_bytes(data.tobytes())
    import subprocess
    subprocess.run([api.CLI_PATH, "-c", "-i", str(src), str(comp)], check=True, timeout=300)
    subprocess.run([api.CLI_PATH, "-c", str(src), str(plain)], check=True, timeout=300)
    assert comp.read_bytes() == plain.read_bytes(), "-i must not change the stream"
    idx = (tmp_path / "c.snp.idx").read_bytes()
    assert idx[:8] == b"SNPIDX1\0" and len(idx) == 24 + 8 * (api.block_count(data.size) + 1)
    subprocess.run([api.CLI_PATH, "-d", "-i", str(comp), str(back)], check=True, timeout=300)
    assert back.read_bytes() == data.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["seg", "tile"])
def test_alternative_decoders(which, tmp_path):
    """Both block decoders, forced with SNAPPY_B200_DECODER (read once per process: csrc/decode.cu) on every
    input, must be bit-exact against the oracle decoder: seg (k_decode_seg, picked above 32 blocks) on the small
    and malformed streams too, tile (k_decode_tile, picked for at most 32 blocks) on the multi-MiB ones too."""
    import subprocess
    import sys
    code = r"""
import sys, os, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, os.path.join(%r, "tests"))
import oracle_lib, streamgen, datasets
from lightweight_snappy_b200 import api
o = oracle_lib.Oracle()
for seed, (total, style) in enumerate([(1, "mixed"), (4095, "copies"), (65537, "copies"), (300001, "bigliteral"), (1 << 20, "mixed"), (2 << 20, "copies")]):
    stream, want = streamgen.make_stream(2000 + seed, total, style)
    assert np.array_equal(o.decompress(stream), want)
    got = api.snappy_decompress(stream)
    assert got.size == want.size and np.array_equal(got, want), (seed, total, style)
for spec in ("corpus:mixed:0:0:7000000", "corpus:lowent:1:0:3000001", "rep:0:200000", "period:3:3:140000", "corpus:random:2:0:200000"):
    data = datasets.gen(spec)
    s = o.compress(data, 0)
    got = api.snappy_decompress(s)
    assert got.size == data.size and np.array_equal(got, data), spec
for bad in (b"\x08\x0cabcd" + bytes([(3 << 2) | 2, 9, 0]), b"\x08\x0cab", b"\x04\x0cabcd\x0cabcd", b"\x20\x0cabcd"):
    try:
        api.snappy_decompress(np.frombuffer(bad, np.uint8))
    except api.SnappyError:
        continue
    raise AssertionError("malformed stream accepted")
print("OK")
"""
    root = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
    env = dict(os.environ, SNAPPY_B200_DECODER=which)
    r = subprocess.run([sys.executable, "-c", code % (root, root)], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0 and "OK" in r.stdout, (r.stdout[-2000:], r.stderr[-3000:])


@pytest.mark.gpu
def test_async_device_api_and_cuda_graph(oracle):
    """SURVEY 8(b): the device-level API only enqueues.  compress + asynchronous index-less decompress are
    captured into ONE CUDA graph and replayed on new data; the replayed stream must equal the oracle's and
    the replayed output the input.  Too few relaxation rounds must be reported (ST_UNRESOLVED), not mis-decoded."""
    import torch
    n = 24 << 20
    codec = api.DeviceCodec(n)
    data = corpus.make_corpus("mixed", n, device="cuda", first_segment=3).clone()
    out = torch.zeros(n, dtype=torch.uint8, device="cuda")
    hdr = len(oracle.varint_encode(n))
    # eager run first (also the warm-up a capture needs), and the compressed size of this data
    codec.compress(data, 0)
    c_bytes = codec.result_stream().numel()
    codec.decompress_async(codec.stream_buf, c_bytes, hdr, n, out)
    codec.check_status()
    assert torch.equal(out, data)
    want = oracle.compress(data.cpu().numpy(), 0)
    _assert_same(codec.result_stream().cpu().numpy(), want, "eager stream")
    # capture
    side = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    out.zero_()
    with torch.cuda.stream(side):
        codec.status.zero_()
        side.synchronize()
        with torch.cuda.graph(g, stream=side):
            codec.compress(data, 0)
            codec.decompress_async(codec.stream_buf, c_bytes, hdr, n, out, zero_status=False)
    # replay on the same buffers after scrambling everything the graph writes
    for _ in range(2):
        out.zero_()
        codec.stream_buf.zero_()
        codec.status.zero_()
        g.replay()
        torch.cuda.synchronize()
        codec.check_status()
        assert int(codec.out_bytes.item()) == c_bytes
        _assert_same(codec.stream_buf[:c_bytes].cpu().numpy(), want, "replayed stream")
        assert torch.equal(out, data), "replayed decode"
    # incompressible data needs far more rounds than 2, and that must be said
    rnd = corpus.make_corpus("random", n, device="cuda")
    codec.compress(rnd, 0)
    cb = codec.result_stream().numel()
    codec.decompress_async(codec.stream_buf, cb, hdr, n, out, max_rounds=2)
    torch.cuda.synchronize()
    assert int(codec.status.item()) & 8, "ST_UNRESOLVED expected"
    with pytest.raises(api.SnappyError):
        codec.check_status()
    codec.decompress_async(codec.stream_buf, cb, hdr, n, out, max_rounds=64)
    codec.check_status()
    assert torch.equal(out, rnd)


@pytest.mark.gpu
@pytest.mark.parametrize("n_devices", [1, 2, 8])
def test_multi_device_host_api(oracle, n_devices):
    """SURVEY 8e behind the C API: block ranges sharded over the visible devices inside the library.  The
    stream and the side index must be byte-identical to the oracle's whatever the device count (more devices
    than the box has are clamped), and both multi-device decoders must invert it."""
    n = (300 << 20) + 70001 if n_devices > 1 else (70 << 20) + 5
    data = corpus.make_corpus("mixed", n, device="cuda", first_segment=11).cpu().numpy()
    want = oracle.compress(data, 0)
    ref_idx, _ = oracle.block_index(want)
    stream, offs = api.compress_host_multi(data, api.MODE_HASH, n_devices, with_index=True)
    _assert_same(stream, want, f"multi-device stream ({n_devices} devices asked, {api.device_count()} present)")
    assert np.array_equal(offs, ref_idx.astype(np.uint64)), "multi-device side index"
    _assert_same(api.decompress_host_multi(want, n_devices), data, "multi-device index-less decode")
    _assert_same(api.decompress_host_multi(want, n_devices, block_offsets=offs), data, "multi-device indexed decode")
    small = data[: 5 << 20]
    _assert_same(api.compress_host_multi(small, api.MODE_BST, n_devices), oracle.compress(small, 1), "multi-device BST")


@pytest.mark.gpu
def test_unframed_foreign_streams(oracle):
    """SURVEY 8f-2: valid raw Snappy whose elements straddle 64 KiB output blocks and whose copies reach
    into earlier blocks (tests/streamgen.py::make_crossing_stream).  The host API must decode it exactly
    like the oracle decoder (the block-parallel path reports FRAMING, the general decoder takes over);
    truly malformed variants of the same streams must still be rejected."""
    import streamgen
    for seed, total in enumerate([70000, 200000, 1 << 20, (3 << 20) + 17]):
        stream, want = streamgen.make_crossing_stream(3000 + seed, total)
        assert np.array_equal(oracle.decompress(stream), want)
        _assert_same(api.snappy_decompress(stream), want, f"crossing stream {seed} ({total} bytes)")
        # cut short / offset beyond the output so far / trailing garbage: errors, not wrong output
        for bad in (stream[:-1], np.concatenate([stream, np.zeros(3, np.uint8)])):
            with pytest.raises(api.SnappyError):
                api.snappy_decompress(bad)
    # a copy that reaches before the start of the output
    bad = np.frombuffer(b"\x90\x4e" + b"\x0cabcd" + bytes([(63 << 2) | 3, 5, 0, 0, 0]) + b"\x00" * 8, np.uint8)
    with pytest.raises(api.SnappyError):
        api.snappy_decompress(bad)


@pytest.mark.gpu
def test_streaming_file_layer(tmp_path, oracle, monkeypatch):
    """The FILE* drop-in layer streams: chunks of whole blocks through three page-locked buffers (reader
    thread / GPU pipeline / writer thread), so memory is bounded by the chunk size.  With a 4 MiB chunk a
    70 MB file goes through ~17 chunks; the stream, the side index and the round trip must not notice.
    Also: a declared size that disagrees with the file (the reference writes the declared one,
    src/snappy_compression.c:417) and an input that ends exactly on a chunk boundary."""
    import subprocess
    monkeypatch.setenv("SNAPPY_B200_FILE_CHUNK_MIB", "4")
    for n in ((70 << 20) + 4321, 8 << 20):
        data = corpus.make_corpus("mixed", n, device="cuda", first_segment=5).cpu().numpy()
        src, comp, back, bst = (tmp_path / x for x in ("in.bin", "c.snp", "back.bin", "c.bsnp"))
        src.write_bytes(data.tobytes())
        env = dict(os.environ)
        subprocess.run([api.CLI_PATH, "-c", "-i", str(src), str(comp)], check=True, timeout=300, env=env)
        got = np.fromfile(comp, np.uint8)
        want = oracle.compress(data, 0)
        _assert_same(got, want, f"streamed -c stream ({n} bytes)")
        idx = np.fromfile(str(comp) + ".idx", np.uint64)
        ref_idx, _ = oracle.block_index(want)
        assert idx[1] == n and idx[2] == api.block_count(n) and np.array_equal(idx[3:], ref_idx.astype(np.uint64))
        subprocess.run([api.CLI_PATH, "-d", str(comp), str(back)], check=True, timeout=300, env=env)
        assert np.array_equal(np.fromfile(back, np.uint8), data)
    small = data[: 3 << 20]
    src.write_bytes(small.tobytes())
    subprocess.run([api.CLI_PATH, "-b", str(src), str(bst)], check=True, timeout=300, env=env)
    _assert_same(np.fromfile(bst, np.uint8), oracle.compress(small, 1), "streamed -b stream")
    # the library call with a wrong declared size: preamble = declared, body = what the file holds
    import ctypes as C
    libc = C.CDLL(None)
    libc.fopen.restype = C.c_void_p
    libc.fopen.argtypes = [C.c_char_p, C.c_char_p]
    libc.fclose.argtypes = [C.c_void_p]
    L = api.lib()
    L.snappy_compress.restype = None
    L.snappy_compress.argtypes = [C.c_void_p, C.c_ulonglong, C.c_void_p]
    fi, fo = libc.fopen(str(src).encode(), b"rb"), libc.fopen(str(comp).encode(), b"wb")
    L.snappy_compress(fi, 12345, fo)
    libc.fclose(fi), libc.fclose(fo)
    got = np.fromfile(comp, np.uint8)
    want = oracle.compress(small, 0)
    hdr = len(oracle.varint_encode(small.size))
    assert got[:2].tobytes() == oracle.varint_encode(12345) and np.array_equal(got[2:], want[hdr:])


@pytest.mark.gpu
def test_second_device_small_bst_input(oracle):
    """ADVICE r1: the opt-in to large dynamic shared memory is per device.  A one-block BST input takes the
    shared-memory table tiers; it must work with cuda:1 current after cuda:0 has already been used (and the
    host contexts are per device, so the two devices do not tear each other's buffers down)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    data = datasets.gen("corpus:text:4:0:1000")
    want = oracle.compress(data, 1)
    with torch.cuda.device(0):
        _assert_same(api.snappy_compress_bst(data), want, "device 0")
    with torch.cuda.device(1):
        _assert_same(api.snappy_compress_bst(data), want, "device 1 (after device 0)")
        _assert_same(api.snappy_decompress(want), data, "device 1 decode")
        big = datasets.gen("corpus:text:4:0:300000")
        _assert_same(api.snappy_compress_bst(big), oracle.compress(big, 1), "device 1, several blocks")
    with torch.cuda.device(0):
        _assert_same(api.snappy_compress(data), oracle.compress(data, 0), "device 0 again")
