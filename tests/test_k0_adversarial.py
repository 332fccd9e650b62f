"""K0 worst cases: streams on which no speculative walk merges into the element chain (tests/k0gen.py), through
every index-less decode path, checked against the strict reference (tests/strict_ref.py).

K0 (csrc/index.cu) resolves the chain of 8 KiB groups by a relaxation whose correct prefix grows by at least one
group per round, so a chain over ngroup groups needs at most ngroup rounds plus one that shows nothing moves.
On these streams it needs about that many, which is what this suite pins down:

  * every entry point decodes them exactly, and K0's block offsets equal the strict block index;
  * DeviceCodec.index needs at most ngroup + 2 rounds, and parity_locked at least ngroup // 2 (the family
    must stay the worst case, or the bound is no longer exercised);
  * decompress_async with exactly the rounds K0 needed decodes, with one fewer it reports ST_UNRESOLVED alone
    and writes nothing;
  * a stream of about 16 800 groups decodes through the synchronous calls.  They used to give up after
    16 384 rounds with ST_UNRESOLVED (reported as a corrupt stream) although the stream is valid.

Sizes put ngroup on the edges of the 16 / 48 / 64 batch schedule of the adaptive mode.  GPU tests run one child
process per setting of SNAPPY_B200_DECODER (the decoder picked by size, and the tile decoder), which the library
reads once per process.
"""
from __future__ import annotations

import json
import os
import subprocess
import sys

import numpy as np
import pytest

import k0gen
import strict_ref

BLOCK, GROUP = 65536, 8192
ST_UNRESOLVED = 8
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TESTS = os.path.join(ROOT, "tests")

NGROUPS = (1, 2, 15, 16, 17, 63, 64, 65, 129, 1000)
SMALL = 65          # cases up to this many groups also run under the tile decoder (<= 32 output blocks)
CAP_NGROUP = 16800  # more than the 16 384 rounds the adaptive mode used to allow


def _make(family, ngroup):
    """(stream, want) of one case: the body has exactly `ngroup` groups."""
    seed = 1000 * (1 + ("parity_locked", "false_kills", "fake_max_literals").index(family)) + ngroup
    if family == "parity_locked":  # the last group (nearly) full; the big ones with short copies, as the cap case
        return k0gen.parity_locked(seed, ngroup * GROUP - 1, max_copy_len=4 if ngroup > 128 else 11)
    if family == "false_kills":    # the last group half full
        return k0gen.false_kills(seed, (ngroup - 1) * GROUP + 4097)
    n_blocks, last = k0gen.fake_size_for(ngroup)
    return k0gen.fake_max_literals(seed, n_blocks, last_bytes=last)


CASES = [(f, g) for g in NGROUPS for f in ("parity_locked", "false_kills", "fake_max_literals")]
CPU_CASES = [(f, g) for f, g in CASES if g <= 129]


def _cid(family, ngroup):
    return f"{family}/{ngroup}"


@pytest.fixture(scope="module")
def cases():
    return {_cid(f, g): _make(f, g) for f, g in CASES}


def _body(stream):
    return stream[strict_ref.varint(stream)[1]:]


# ---------------------------------------------------------------------------------------------- CPU part
def test_generators_are_deterministic_and_sized(cases):
    for (f, g) in CASES:
        stream, want = cases[_cid(f, g)]
        assert k0gen.ngroup_of(_body(stream).size) == g, (f, g)
        assert strict_ref.varint(stream)[0] == want.size
    for f, g in (("parity_locked", 17), ("false_kills", 17), ("fake_max_literals", 17)):
        s2, w2 = _make(f, g)
        s1, w1 = cases[_cid(f, g)]
        assert np.array_equal(s1, s2) and np.array_equal(w1, w2)


@pytest.mark.parametrize("family,ngroup", CPU_CASES, ids=[_cid(f, g) for f, g in CPU_CASES])
def test_strict_reference_and_oracle_agree(cases, oracle, family, ngroup):
    stream, want = cases[_cid(family, ngroup)]
    out, why = strict_ref.strict_decode(stream)
    assert out == want.tobytes(), why
    index, ng = k0gen.layout(stream)  # valid, framed in 64 KiB blocks
    assert ng == ngroup and len(index) == (want.size + BLOCK - 1) // BLOCK + 1
    assert np.array_equal(oracle.decompress(stream), want)
    assert [int(x) for x in oracle.block_index(stream)[0]] == index


@pytest.mark.parametrize("ngroup", [1, 2, 16, 65])
def test_parity_locked_walks_never_merge(cases, ngroup):
    stream, _ = cases[_cid("parity_locked", ngroup)]
    body = _body(stream)
    assert np.all(body[2::2] & 3 == 1) and body[0] == 1 << 2  # every even byte after the first is a copy-1 tag
    chain = k0gen.chain_starts(stream)
    assert chain[0] == 0 and np.all(chain[1:] % 2 == 1)
    r = k0gen.walk_report(stream, max_elems=4096)
    assert r["merged"][0] and not r["merged"][1:].any()
    assert np.all(r["longest"][1:] == 2)


def test_parity_locked_big_stream_is_locked(cases):
    """The structural property on the largest case (the walk model would be slow there)."""
    stream, want = cases[_cid("parity_locked", 1000)]
    body = _body(stream)
    assert np.all(body[2::2] & 3 == 1) and body.size % 2 == 1
    assert want.size / stream.size > 1.8  # max_copy_len=4: about 2 output bytes per stream byte


@pytest.mark.parametrize("ngroup", [16, 65, 129])
def test_false_kills_jump_far(cases, ngroup):
    stream, _ = cases[_cid("false_kills", ngroup)]
    body = _body(stream)
    fakes = np.isin(body[2::2], k0gen.FAKE_TAGS)
    assert fakes.sum() >= ngroup  # about one per 768 bytes
    r = k0gen.walk_report(stream, max_elems=4096)
    assert np.all(r["steps"][1:] > 0)  # no grid point after the first starts on the chain
    assert (r["longest"] >= GROUP).sum() >= 4  # some wrong-phase walks jump over whole groups ...
    assert r["merged"][1:].any() and not r["merged"][1:].all()  # ... and land on either phase
    assert (r["end"] >= r["body"]).any()  # and some leave the body (0xf8 / 0xfc: megabyte lengths)


@pytest.mark.parametrize("ngroup", [15, 65, 129])
def test_fake_max_literals_chains_run_to_the_end(cases, ngroup):
    stream, want = cases[_cid("fake_max_literals", ngroup)]
    assert stream.size // 4 >= want.size // 5  # >= 80 %: k_group_init's literal scan is on
    hdr = strict_ref.varint(stream)[1]
    index, _ = k0gen.layout(stream)
    n_blocks = len(index) - 1
    assert n_blocks >= 2
    deltas = [d for d in (7, 2000, 33333, 65530)]
    starts = [index[0] - hdr + 3 + d for d in deltas]  # the fake headers in block 0's payload
    assert all(bytes(_body(stream)[s:s + 3]) == b"\xf4\xff\xff" for s in starts)
    r = k0gen.walk_report(stream, starts=starts, max_elems=10 * n_blocks)
    assert not r["merged"].any()
    assert np.all(r["longest"] == k0gen.MAX_LITERAL)  # fake after fake ...
    assert np.all(r["end"] >= r["body"])  # ... until the walk leaves the body
    last = want.size - (n_blocks - 1) * BLOCK
    assert np.all(r["steps"] == [n_blocks if d + 3 <= last else n_blocks - 1 for d in deltas])


def test_cap_case_exceeds_the_old_round_cap():
    """The stream the GPU cap test decodes: valid (oracle), about 2 output bytes per stream byte, and more
    groups than the old cap of 16 384 rounds plus a batch."""
    import oracle_lib
    stream, want = k0gen.parity_locked(16800, CAP_NGROUP * GROUP - 1, max_copy_len=4)
    assert k0gen.ngroup_of(_body(stream).size) == CAP_NGROUP > (1 << 14) + 2 + 64
    assert np.all(_body(stream)[2::2] & 3 == 1)
    assert np.array_equal(oracle_lib.Oracle().decompress(stream), want)


# ---------------------------------------------------------------------------------------------- GPU part
@pytest.fixture(scope="module")
def matrix(tmp_path_factory, cases, oracle):
    """The cases and what the strict reference says about them, written before any GPU call."""
    arrays, meta = {}, []
    for f, g in CASES:
        stream, want = cases[_cid(f, g)]
        if g <= 129:
            index, _ = k0gen.layout(stream)
        else:  # the strict reference is slow at 8 MiB; these are checked against it on the CPU at smaller sizes
            index = [int(x) for x in oracle.block_index(stream)[0]]
            assert np.array_equal(oracle.decompress(stream), want)
        key = f"c{len(meta)}"
        arrays[key], arrays[key + "w"] = stream, want
        meta.append({"id": _cid(f, g), "key": key, "family": f, "ngroup": g, "index": index,
                     "hdr": strict_ref.varint(stream)[1]})
    d = tmp_path_factory.mktemp("k0adv")
    np.savez(d / "streams.npz", **arrays)
    (d / "meta.json").write_text(json.dumps(meta))
    return d


_CHILD = r"""
import json, os, subprocess, sys, tempfile
import numpy as np, torch
sys.path.insert(0, %(root)r)
from lightweight_snappy_b200 import api
ST_UNRESOLVED, SENTINEL = 8, 0xA5
d = sys.argv[1]
max_ngroup = int(sys.argv[2])
arr = np.load(os.path.join(d, "streams.npz"))
meta = json.load(open(os.path.join(d, "meta.json")))
with_cli = os.environ.get("K0ADV_CLI") == "1"
two_gpus = torch.cuda.device_count() >= 2
fails, rounds = [], {}
tmp = tempfile.mkdtemp()

def fail(cid, call, what):
    fails.append([cid, call, what])

def host(cid, call, fn, want, env=None):
    print(cid, call, flush=True)
    saved = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    try:
        got = fn()
        if got.size != want.size or not np.array_equal(got, want):
            fail(cid, call, "wrong output")
    except api.SnappyError as x:
        fail(cid, call, "valid stream rejected: " + str(x))
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v

for e in meta:
    if e["ngroup"] > max_ngroup:
        continue
    cid, stream, want = e["id"], arr[e["key"]], arr[e["key"] + "w"]
    total, hdr, ng = want.size, e["hdr"], e["ngroup"]
    host(cid, "snappy_decompress", lambda: api.snappy_decompress(stream), want)
    host(cid, "decompress_host(1 MiB pieces)", lambda: api.decompress_host(stream), want,
         {"SNAPPY_B200_PIECE_MIB": "1", "SNAPPY_B200_PIECE_START_MIB": "1"})
    if two_gpus:
        host(cid, "host_multi(2)", lambda: api.decompress_host_multi(stream, 2), want)
    codec = api.DeviceCodec(max(total, stream.size))
    d_stream = torch.from_numpy(np.concatenate([stream, np.zeros(64, np.uint8)])).cuda()
    want_t = torch.from_numpy(want).cuda()
    out = torch.empty(total, dtype=torch.uint8, device="cuda")
    nb = api.block_count(total)
    index = torch.tensor(e["index"], dtype=torch.int64, device="cuda")
    offs = torch.zeros(nb + 1, dtype=torch.int64, device="cuda")

    def device(call, fn, check_out=True, check_offs=True):
        print(cid, call, flush=True)
        out.fill_(SENTINEL)
        offs.zero_()
        try:
            fn()
            torch.cuda.synchronize()
        except api.SnappyError as x:
            fail(cid, call, "valid stream rejected by the call: " + str(x))
            return None
        st = int(codec.status.item())
        if st != 0:
            fail(cid, call, "status 0x%%x" %% st)
        elif check_out and not torch.equal(out, want_t):
            fail(cid, call, "status 0 but wrong output")
        elif check_offs and not torch.equal(offs, index):
            fail(cid, call, "K0 offsets differ from the strict index")
        return st

    device("decompress", lambda: codec.decompress(d_stream, stream.size, hdr, total, out, offs))
    if device("index", lambda: codec.index(d_stream, stream.size, hdr, total, offs), check_out=False) is not None:
        r = api.index_rounds()
        rounds[cid] = r
        if r > ng + 2:
            fail(cid, "index", "%%d rounds for %%d groups: more than ngroup + 2" %% (r, ng))
        if e["family"] == "parity_locked" and r < ng // 2:
            fail(cid, "index", "%%d rounds for %%d groups: parity_locked is no longer the worst case" %% (r, ng))
        if 2 <= r <= 64:
            device("async(max_rounds=R)", lambda: codec.decompress_async(d_stream, stream.size, hdr, total, out, offs,
                                                                         max_rounds=r))
            print(cid, "async(max_rounds=R-1)", flush=True)
            out.fill_(SENTINEL)
            codec.decompress_async(d_stream, stream.size, hdr, total, out, offs, max_rounds=r - 1)
            torch.cuda.synchronize()
            st = int(codec.status.item())
            if st != ST_UNRESOLVED:
                fail(cid, "async(max_rounds=R-1)", "status 0x%%x, not ST_UNRESOLVED alone" %% st)
            if not bool((out == SENTINEL).all()):
                fail(cid, "async(max_rounds=R-1)", "unresolved, but the output buffer was written")
    print(cid, "decompress_indexed", flush=True)
    out.fill_(SENTINEL)
    codec.decompress_indexed(d_stream, index, total, out)
    torch.cuda.synchronize()
    st = int(codec.status.item())
    if st != 0 or not torch.equal(out, want_t):
        fail(cid, "decompress_indexed", "status 0x%%x, output %%s" %% (st, "exact" if torch.equal(out, want_t) else "wrong"))
    if with_cli:
        src, dst = os.path.join(tmp, "in.snp"), os.path.join(tmp, "out.bin")
        stream.tofile(src)
        print(cid, "cli", flush=True)
        r = subprocess.run([api.CLI_PATH, "-d", src, dst], capture_output=True, text=True)
        if r.returncode != 0 or not np.array_equal(np.fromfile(dst, np.uint8), want):
            fail(cid, "cli", "exit %%d %%s" %% (r.returncode, r.stderr[-200:]))
    del codec, d_stream, want_t, out
print("ROUNDS " + json.dumps(rounds))
print("FAILS " + json.dumps(fails))
"""

SETTINGS = {
    "default": ({"K0ADV_CLI": "1"}, max(NGROUPS)),
    "tile": ({"SNAPPY_B200_DECODER": "tile"}, SMALL),
}
_SWITCHES = ("SNAPPY_B200_DECODER", "SNAPPY_B200_PIECE_MIB", "SNAPPY_B200_PIECE_START_MIB",
             "SNAPPY_B200_PIECE_GROWTH", "SNAPPY_B200_DEVICES")


def _run_child(code, args, env_over, timeout=1800):
    env = {k: v for k, v in os.environ.items() if k not in _SWITCHES}
    env.update(env_over)
    return subprocess.run([sys.executable, "-c", code] + args, capture_output=True, text=True, timeout=timeout, env=env)


@pytest.mark.gpu
@pytest.mark.parametrize("setting", list(SETTINGS))
def test_k0_adversarial_matrix(matrix, setting):
    """Every case through snappy_decompress (default and 1 MiB pieces), decompress_host_multi over two devices
    (when there are two), DeviceCodec.decompress / index / decompress_indexed, the async round boundary and,
    under the default setting, `snappy_b200 -d`."""
    env, max_ngroup = SETTINGS[setting]
    r = _run_child(_CHILD % {"root": ROOT}, [str(matrix), str(max_ngroup)], env)
    lines = r.stdout.strip().splitlines()
    fails = [json.loads(ln[6:]) for ln in lines if ln.startswith("FAILS ")]
    rounds = [json.loads(ln[7:]) for ln in lines if ln.startswith("ROUNDS ")]
    assert r.returncode == 0 and fails, (f"child ended with {r.returncode}; last call: "
                                         f"{lines[-1] if lines else None}", r.stderr[-3000:])
    print(f"\n[{setting}] K0 rounds (DeviceCodec.index) per case:")
    for cid, n in rounds[0].items():
        print(f"  {cid:24s} ngroup {cid.split('/')[1]:>5s}  rounds {n}")
    assert fails[0] == [], json.dumps(fails[0][:40], indent=0)


_CHILD_CAP = r"""
import json, os, subprocess, sys, tempfile, time
import numpy as np, torch
sys.path.insert(0, %(root)r); sys.path.insert(0, %(tests)r)
from lightweight_snappy_b200 import api
import k0gen, oracle_lib
ngroup = %(ngroup)d
t0 = time.perf_counter()
stream, want = k0gen.parity_locked(16800, ngroup * 8192 - 1, max_copy_len=4)
oracle = oracle_lib.Oracle()
assert np.array_equal(oracle.decompress(stream), want), "generator and oracle disagree"
index = [int(x) for x in oracle.block_index(stream)[0]]
hdr = len(k0gen.varint(want.size))
total = want.size
assert k0gen.ngroup_of(stream.size - hdr) == ngroup
print("stream %%d bytes, output %%d bytes, %%d groups, built in %%.1f s" %% (stream.size, total, ngroup,
      time.perf_counter() - t0), flush=True)
fails, report = [], {"ngroup": ngroup, "stream_bytes": int(stream.size), "output_bytes": int(total)}

def timed(name, fn):
    print(name, flush=True)
    t = time.perf_counter()
    try:
        r = fn()
        torch.cuda.synchronize()
    except api.SnappyError as x:
        fails.append([name, "valid stream rejected: " + str(x)])
        r = None
    report[name] = {"seconds": round(time.perf_counter() - t, 3)}
    return r

codec = api.DeviceCodec(total)
d_stream = torch.from_numpy(np.concatenate([stream, np.zeros(64, np.uint8)])).cuda()
want_t = torch.from_numpy(want).cuda()
index_t = torch.tensor(index, dtype=torch.int64, device="cuda")
out = torch.empty(total, dtype=torch.uint8, device="cuda")
offs = torch.zeros(len(index), dtype=torch.int64, device="cuda")
for call in ("DeviceCodec.index", "DeviceCodec.decompress"):
    out.zero_(); offs.zero_()
    if call == "DeviceCodec.index":
        timed(call, lambda: codec.index(d_stream, stream.size, hdr, total, offs))
    else:
        timed(call, lambda: codec.decompress(d_stream, stream.size, hdr, total, out, offs))
    st, r = int(codec.status.item()), api.index_rounds()
    report[call].update(status=st, rounds=r)
    if st != 0:
        fails.append([call, "status 0x%%x after %%d rounds" %% (st, r)])
        continue
    if not torch.equal(offs, index_t):
        fails.append([call, "K0 offsets differ from the oracle's block index"])
    if call == "DeviceCodec.decompress" and not torch.equal(out, want_t):
        fails.append([call, "wrong output"])
    if not ngroup // 2 <= r <= ngroup + 2:
        fails.append([call, "%%d rounds for %%d groups" %% (r, ngroup)])
del d_stream, want_t, index_t, out, offs, codec
torch.cuda.empty_cache()
tmp = tempfile.mkdtemp()
src, dst = os.path.join(tmp, "in.snp"), os.path.join(tmp, "out.bin")
stream.tofile(src)
p = timed("snappy_b200 -d", lambda: subprocess.run([api.CLI_PATH, "-d", src, dst], capture_output=True, text=True))
if p is not None and (p.returncode != 0 or not np.array_equal(np.fromfile(dst, np.uint8), want)):
    fails.append(["snappy_b200 -d", "exit %%d %%s" %% (p.returncode, p.stderr[-300:])])
os.remove(dst)
if torch.cuda.device_count() >= 2:
    got = timed("decompress_host_multi(2)", lambda: api.decompress_host_multi(stream, 2))
    if got is not None and not np.array_equal(got, want):
        fails.append(["decompress_host_multi(2)", "wrong output"])
os.environ.update(SNAPPY_B200_PIECE_MIB="256", SNAPPY_B200_PIECE_START_MIB="256")
got = timed("snappy_decompress(256 MiB pieces)", lambda: api.snappy_decompress(stream))
if got is not None and not np.array_equal(got, want):
    fails.append(["snappy_decompress(256 MiB pieces)", "wrong output"])
print("CAP " + json.dumps(report))
print("FAILS " + json.dumps(fails))
"""


@pytest.mark.gpu
def test_k0_cap_case():
    """parity_locked with about 16 800 groups (138 MB of stream, 275 MB of output) through DeviceCodec.index and
    .decompress, `snappy_b200 -d`, decompress_host_multi over two devices (when there are two) and
    snappy_decompress with one 256 MiB K0 region.  Every call must decode it; K0 needs about one round per group."""
    r = _run_child(_CHILD_CAP % {"root": ROOT, "tests": TESTS, "ngroup": CAP_NGROUP}, [], {})
    lines = r.stdout.strip().splitlines()
    fails = [json.loads(ln[6:]) for ln in lines if ln.startswith("FAILS ")]
    report = [json.loads(ln[4:]) for ln in lines if ln.startswith("CAP ")]
    assert r.returncode == 0 and fails, (f"child ended with {r.returncode}; last call: "
                                         f"{lines[-1] if lines else None}", r.stderr[-3000:])
    print("\n" + json.dumps(report[0], indent=1))
    assert fails[0] == [], json.dumps(fails[0], indent=0)
