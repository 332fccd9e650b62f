"""k_decode_seg's pointer doubling over lanes, which resolves a copy whose source byte is produced in the
same 32-byte round, on streams full of short copy chains, against the oracle decoder and the generator's
own output.  Every stream has more than 32 blocks, so the segment decoder runs and not the tile decoder."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

BLOCK = 65536
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _varint(n: int) -> bytes:
    out = bytearray()
    while n >= 0x80:
        out.append((n & 0x7F) | 0x80)
        n >>= 7
    out.append(n)
    return bytes(out)


def _literal(data: bytes) -> bytes:
    m = len(data) - 1
    if m < 60:
        return bytes([m << 2]) + data
    return bytes([60 << 2, m]) + data if m < 256 else bytes([61 << 2]) + m.to_bytes(2, "little") + data


def _copy(length: int, off: int, copy4: bool) -> bytes:
    if copy4:
        return bytes([((length - 1) << 2) | 3]) + off.to_bytes(4, "little")
    if 4 <= length <= 11 and off < 2048:
        return bytes([((off >> 8) << 5) | ((length - 4) << 2) | 1, off & 0xFF])
    return bytes([((length - 1) << 2) | 2]) + off.to_bytes(2, "little")


def make_chain_stream(seed: int, total: int, p_long: float, p_copy4: float) -> tuple[np.ndarray, np.ndarray]:
    """Blocks made mostly of copies with offsets 1..40 and lengths 4..64 (overlapping and not), so that
    most rounds hold chains of in-round sources, cut by literals of 64 bytes or more (p_long) and
    copy-4 elements (p_copy4), both of which end a run.  Returns (stream, expected output)."""
    rng = np.random.default_rng(seed)
    out = bytearray()
    stream = bytearray(_varint(total))
    while len(out) < total:
        block_len = min(BLOCK, total - len(out))
        base = len(out)
        while len(out) - base < block_len:
            produced, room = len(out) - base, block_len - (len(out) - base)
            r = rng.random()
            if produced == 0 or r < 0.12:
                n = int(rng.integers(1, 17))
            elif r < 0.12 + p_long:
                n = int(rng.integers(64, 300))
            else:
                n = 0
            if n:
                data = rng.integers(0, 256, min(n, room), dtype=np.uint8).tobytes()
                stream += _literal(data)
                out += data
                continue
            n = min(int(rng.integers(4, 65)), room)
            off = int(rng.integers(1, min(produced, 40) + 1))
            stream += _copy(n, off, rng.random() < p_copy4)
            start = len(out) - off
            period = bytes(out[start:])
            out += (period * (n // off + 1))[:n]  # write_copy: an overlapping copy repeats the last `off` bytes
    return np.frombuffer(bytes(stream), np.uint8).copy(), np.frombuffer(bytes(out), np.uint8).copy()


CASES = [  # (seed, total bytes, p_long, p_copy4)
    (1, 33 * BLOCK, 0.0, 0.0),          # one run per segment: chains cross rounds and segment (run) ends
    (2, 40 * BLOCK + 45, 0.03, 0.0),    # long literals cut runs; the last block ends mid-round
    (3, 36 * BLOCK + 1000, 0.0, 0.05),  # copy-4 elements cut runs
    (4, 34 * BLOCK + 17, 0.05, 0.05),   # both, short partial rounds everywhere
]

_CHILD = r"""
import sys, os, numpy as np, torch
sys.path.insert(0, %r)
from lightweight_snappy_b200 import api
d = np.load(sys.argv[1])
for i in range(len(d.files) // 2):
    stream, want = d["s%%d" %% i], d["w%%d" %% i]
    got = api.snappy_decompress(stream)  # host API: K0 + segment decoder
    assert got.size == want.size and np.array_equal(got, want), ("host", i, int(np.argmax(got != want)))
    n = want.size
    nb = api.block_count(n)
    assert nb > 32
    hdr = 1
    while n >> (7 * hdr):
        hdr += 1
    codec = api.DeviceCodec(n)
    d_stream = torch.from_numpy(np.concatenate([stream, np.zeros(64, np.uint8)])).cuda()
    out = torch.zeros(n, dtype=torch.uint8, device="cuda")
    codec.decompress(d_stream, stream.size, hdr, n, out, torch.zeros(nb + 1, dtype=torch.int64, device="cuda"))
    codec.check_status()
    got = out.cpu().numpy()
    assert np.array_equal(got, want), ("device", i, int(np.argmax(got != want)))
print("OK")
"""


@pytest.fixture(scope="module")
def chain_streams(tmp_path_factory, oracle):
    arrays = {}
    for i, (seed, total, p_long, p_copy4) in enumerate(CASES):
        stream, want = make_chain_stream(seed, total, p_long, p_copy4)
        assert np.array_equal(oracle.decompress(stream), want), f"generator and oracle disagree on case {i}"
        arrays[f"s{i}"], arrays[f"w{i}"] = stream, want
    path = tmp_path_factory.mktemp("inround") / "streams.npz"
    np.savez(path, **arrays)
    return path


def test_inround_chains(chain_streams):
    """Decodes in a process of its own, with the decoder picked by input size (SNAPPY_B200_DECODER unset)."""
    env = dict(os.environ)
    env.pop("SNAPPY_B200_DECODER", None)
    r = subprocess.run([sys.executable, "-c", _CHILD % ROOT, str(chain_streams)], capture_output=True, text=True,
                       timeout=600, env=env)
    assert r.returncode == 0 and "OK" in r.stdout, (r.stdout[-2000:], r.stderr[-3000:])


@pytest.mark.parametrize("kind", ["text", "lowent"])
def test_device_decode_64mib(kind):
    """The corpora whose rounds hold the most in-round sources, compressed and decoded on the device."""
    import torch
    from lightweight_snappy_b200 import api, corpus
    n = 64 << 20
    data = corpus.make_corpus(kind, n, device="cuda")
    codec = api.DeviceCodec(n)
    codec.compress(data, api.MODE_HASH)
    stream = codec.result_stream().clone()
    hdr = 1
    while n >> (7 * hdr):
        hdr += 1
    out = torch.zeros(n, dtype=torch.uint8, device="cuda")
    codec.decompress(stream, stream.numel(), hdr, n, out, torch.zeros(api.block_count(n) + 1, dtype=torch.int64,
                                                                      device="cuda"))
    codec.check_status()
    assert torch.equal(out, data)
