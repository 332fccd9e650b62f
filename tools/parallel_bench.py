"""MODE_PARALLEL against MODE_HASH on one GPU.

    python tools/parallel_bench.py [--mib 1024] [--reps 5] [--out profiles/r05_parallel.json]

  compress_ms_per_gib    snappy_b200_compress_device on --mib of each corpus class, CUDA events, warm-up, then the
                         median of --reps runs with the two modes alternating; compressed bytes for both
  decompress_ms_per_gib  the same streams through snappy_b200_decompress_device (K0 + block decode), alternating
  host_ms                snappy_b200_compress_host (pageable buffers, wall clock around the synchronous call) at
                         4 KiB, 64 KiB, 1 MiB and 16 MiB of mixed data, both modes alternating, median of 20
  kernels_ms             torch.profiler, after the timed runs: the kernels of one MODE_PARALLEL compress of the mixed
                         corpus (k_par_cand, k_par_walk, k_emit, k_scan_sizes, k_gather)
The input is larger than L2 at the default size.  The card's name and power limit are read in the same run and written
beside the numbers, and the SM clock is read again right after each class's timed compress loop, while the card is
still at its working clock (sm_clock_mhz_after_compress).
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np
import torch

from lightweight_snappy_b200 import api, corpus

ap = argparse.ArgumentParser()
ap.add_argument("--mib", type=int, default=1024)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--out", default="profiles/r05_parallel.json")
a = ap.parse_args()
assert torch.cuda.is_available(), "parallel_bench measures on the GPU"
n = a.mib << 20
gib = n / (1 << 30)
MODES = ((api.MODE_HASH, "hash"), (api.MODE_PARALLEL, "parallel"))


def alternating(fns, reps):
    """fns: name -> callable (device work on the current stream).  Warm-up, then reps rounds in turn."""
    for fn in fns.values():
        fn()
    torch.cuda.synchronize()
    ts = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts[k].append(e0.elapsed_time(e1))
    return {k: float(np.median(v)) for k, v in ts.items()}


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_sm_clock_max_sm_clock": smi[0] if smi else None,
       "mib": a.mib, "reps": a.reps, "statistic": "median"}

codec = api.DeviceCodec(n)
streams = {m: torch.empty(codec.comp_capacity, dtype=torch.uint8, device="cuda") for m, _ in MODES}
out = torch.empty(n, dtype=torch.uint8, device="cuda")
body = 1  # the stream's body starts after the varint of n
while n >> (7 * body):
    body += 1


def sm_clock():
    r = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip()
    return r.splitlines()[0] if r else None


comp, dec, sizes, clocks = {}, {}, {}, {}
for kind in ("text", "lowent", "random", "mixed"):
    data = corpus.make_corpus(kind, n, device="cuda")
    t = alternating({name: (lambda m=m: codec.compress(data, m)) for m, name in MODES}, a.reps)
    clocks[kind] = sm_clock()
    comp[kind] = {k: v / gib for k, v in t.items()}
    lens = {}
    for m, name in MODES:
        codec.compress(data, m)
        lens[m] = int(codec.result_stream().numel())
        streams[m][:lens[m]].copy_(codec.stream_buf[:lens[m]])
    sizes[kind] = {name: lens[m] for m, name in MODES}
    sizes[kind]["parallel_over_hash"] = lens[api.MODE_PARALLEL] / lens[api.MODE_HASH]
    t = alternating({name: (lambda m=m: codec.decompress(streams[m], lens[m], body, n, out)) for m, name in MODES},
                    a.reps)
    dec[kind] = {k: v / gib for k, v in t.items()}
    dec[kind]["parallel_over_hash"] = t["parallel"] / t["hash"]
    codec.decompress(streams[api.MODE_PARALLEL], lens[api.MODE_PARALLEL], body, n, out)
    codec.check_status()
    assert torch.equal(out, data), f"{kind}: the parallel-mode stream does not decode to the input"
    del data
res["compress_ms_per_gib"] = comp
res["sm_clock_mhz_after_compress"] = clocks
res["compressed_bytes"] = sizes
res["decompress_ms_per_gib"] = dec

host = {}
mixed = corpus.make_corpus("mixed", 16 << 20).numpy()
for size in (4 << 10, 64 << 10, 1 << 20, 16 << 20):
    buf = np.ascontiguousarray(mixed[:size])
    out_h = np.empty(api.max_compressed_bytes(size) + 16, np.uint8)
    for m, _ in MODES:
        for _ in range(3):
            api.compress_host(buf, m, out=out_h)
    ts = {name: [] for _, name in MODES}
    for _ in range(20):
        for m, name in MODES:
            t0 = time.perf_counter()
            api.compress_host(buf, m, out=out_h)
            ts[name].append((time.perf_counter() - t0) * 1e3)
    host[f"{size >> 10}KiB"] = {k: float(np.median(v)) for k, v in ts.items()}
res["host_ms"] = host

from torch.profiler import ProfilerActivity, profile  # noqa: E402

data = corpus.make_corpus("mixed", n, device="cuda")
codec.compress(data, api.MODE_PARALLEL)
torch.cuda.synchronize()
names = ["k_par_cand", "k_par_walk", "k_emit", "k_scan_sizes", "k_gather"]
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(a.reps):
        codec.compress(data, api.MODE_PARALLEL)
    torch.cuda.synchronize()
tot = {k: 0.0 for k in names}
for e in prof.key_averages():
    for k in names:
        if k in e.key:
            tot[k] += e.device_time_total / 1e3 / a.reps
res["kernels_ms"] = {"corpus": "mixed", "mode": "parallel", **tot}

os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
with open(a.out, "w") as f:
    json.dump(res, f, indent=1)
print(json.dumps(res, indent=1))
