"""Cost of the framing format on one GPU: 1 GiB of the mixed corpus, warm-up, then the median of --reps runs.

    python tools/frame_bench.py [--mib 1024] [--reps 5] [--out profiles/r04_frame.json]

  compress_device_ms     snappy_b200_compress_device vs snappy_b200_frame_compress_device, hash and BST (CUDA events)
  kernels_ms             from torch.profiler (a run of its own): k_crc32c_chunks per GiB of input in the framed
                         compressor; the framed decode kernels (k_frame_decode + k_crc32c_chunks, in
                         frame_decompress_host) vs snappy_b200_decompress_device_indexed (k_decode_warp) on the same
                         data
  host_decompress_ms     pinned host buffers, wall clock around the synchronous calls: frame_decompress_host vs
                         decompress_host_indexed vs decompress_host
  framed_over_raw_size   framed stream bytes / raw stream bytes
The card's name and power limit are read in the same run and written beside the numbers.
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
ap.add_argument("--out", default="profiles/r04_frame.json")
a = ap.parse_args()
assert torch.cuda.is_available(), "frame_bench measures on the GPU"
n = a.mib << 20
gib = n / (1 << 30)


def ev_median(fn):
    fn()
    ts = []
    for _ in range(a.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts))


def wall_median(fn):
    fn()
    ts = []
    for _ in range(a.reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def kernel_ms(fn, names):
    """Summed CUDA time of the kernels whose name contains one of `names`, per call (profiled run)."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(a.reps):
            fn()
        torch.cuda.synchronize()
    tot = {k: 0.0 for k in names}
    for e in prof.key_averages():
        for k in names:
            if k in e.key:
                tot[k] += e.device_time_total / 1e3  # us -> ms
    return {k: v / a.reps for k, v in tot.items()}


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "mib": a.mib, "corpus": "mixed",
       "reps": a.reps, "statistic": "median"}

data = corpus.make_corpus("mixed", n, device="cuda")
codec = api.DeviceCodec(n)
comp = {}
for mode, mname in ((0, "hash"), (1, "bst")):
    comp[f"raw_{mname}"] = ev_median(lambda: codec.compress(data, mode))
    comp[f"framed_{mname}"] = ev_median(lambda: codec.compress_framed(data, mode))
res["compress_device_ms"] = comp
codec.compress(data, 0)
raw_bytes = codec.result_stream().numel()
codec.compress_framed(data, 0)
framed_dev = codec.result_stream().cpu().numpy()
res["framed_over_raw_size"] = framed_dev.size / raw_bytes

host = data.cpu().numpy()
del codec
torch.cuda.empty_cache()
raw, offs = api.compress_host_indexed(host, 0)
framed = api.compress_framed(host, 0)
assert np.array_equal(framed, framed_dev), "host and device framed streams differ"
pin_raw = torch.from_numpy(raw).pin_memory().numpy()
pin_framed = torch.from_numpy(framed).pin_memory().numpy()
pin_out = torch.empty(n, dtype=torch.uint8).pin_memory().numpy()
assert np.array_equal(api.decompress_framed(pin_framed, out=pin_out), host)
assert np.array_equal(api.decompress_host_indexed(pin_raw, offs, out=pin_out), host)
res["host_decompress_ms"] = {
    "frame_decompress_host": wall_median(lambda: api.decompress_framed(pin_framed, out=pin_out)),
    "decompress_host_indexed": wall_median(lambda: api.decompress_host_indexed(pin_raw, offs, out=pin_out)),
    "decompress_host": wall_median(lambda: api.decompress_host(pin_raw, out=pin_out)),
}

dev_in = data
codec = api.DeviceCodec(n)
dev_out = torch.empty(n, dtype=torch.uint8, device="cuda")
codec.compress(dev_in, 0)
k_idec = kernel_ms(lambda: codec.decompress_indexed(codec.stream_buf, codec.block_offsets, n, dev_out), ["k_decode_warp"])
codec.check_status()
assert torch.equal(dev_out, dev_in)
k_comp = kernel_ms(lambda: codec.compress_framed(dev_in, 0), ["k_crc32c_chunks"])
k_fdec = kernel_ms(lambda: api.decompress_framed(pin_framed, out=pin_out), ["k_frame_decode", "k_crc32c_chunks"])
res["kernels_ms"] = {
    "k_crc32c_chunks_per_gib_compress": k_comp["k_crc32c_chunks"] / gib,
    "framed_decode_k_frame_decode": k_fdec["k_frame_decode"],
    "framed_decode_k_crc32c_chunks": k_fdec["k_crc32c_chunks"],
    "framed_decode_total": k_fdec["k_frame_decode"] + k_fdec["k_crc32c_chunks"],
    "device_indexed_decode_k_decode_warp": k_idec["k_decode_warp"],
}
os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
with open(a.out, "w") as f:
    json.dump(res, f, indent=1)
print(json.dumps(res, indent=1))
