#!/usr/bin/env python
"""bench.py -- throughput of the Snappy hot path on B200 (BASELINE.json configs[1] and [2]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A step is one pass of the hot path over one batch: the 1 GiB synthetic *mixed* corpus
(text-like / low-entropy / random in 1 MiB segments, SURVEY.md 8d) per GPU.

  value            decompression of the index-less reference-format stream, device resident:
                   uncompressed bytes of all ranks / max-over-ranks CUDA-event time of K steps
                   (each step = K0 boundary discovery + block decode)
  compress{}       the same for hash-table compression (configs[2]), timed in the same run
  e2e              the same metric through the host-buffer C-ABI call (pinned host buffers,
                   H2D + D2H inside the timed region)
  roofline         dominant kernel (block decode): (C + U) / its own CUDA-event time vs the
                   measured HBM copy bandwidth in MEASURED_PEAKS.json
  cpu_baseline     the reference's CPU decoder (oracle/_ref when built, else the oracle port)
                   on a bounded sample of the same corpus, one process per host core

Multi-GPU: one process per GPU under torchrun, blocks partitioned by rank (each rank owns its
own 1 GiB of corpus: weak scaling), no collective on the data path; NCCL only carries the
barrier and the max-over-ranks of the timings.

`--impl reference` times the reference's own CPU implementation (all host cores) on a bounded
sample of the same workload and prints the same JSON line with "impl": "reference".

`--dump-outputs DIR` writes, on rank 0, what each timed device leg returned in its last step
(decompress: output bytes + block offsets; compress and BST: stream + block offsets) as
DIR/<leg>_<array>.npy, so that two builds can be compared output for output on the same seeded
inputs.  Byte arrays are stored as float32 values at fixed, seeded positions (<leg>_<array>_sample)
plus float64 byte sums of every 64 KiB chunk (<leg>_<array>_chunk_sums); offsets as float64.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

GIB = 1 << 30
SEED = 20261018
METRIC = "decompress GB/s (uncompressed)"
DECODE_KERNEL = "k_decode_seg (+ k_copy_literal_blocks)"
DUMP_SAMPLE = 1 << 21       # sampled positions per byte array (8 MiB as float32)
DUMP_MAX_ENTRIES = 1 << 19  # longer offset / chunk-sum arrays are sampled too (4 MiB as float64)
DUMP_LIMIT = 64 << 20       # all dumped files together


# ------------------------------------------------------------------------------ CPU baseline
def _cpu_worker(args):
    """One host core: generate a shard of the corpus, then time the CPU codec on it."""
    shard, n_bytes, use_ref, kind, mode, cpu = args
    import numpy as np
    import torch
    torch.set_num_threads(1)
    try:  # one worker per core, pinned: the aggregate stops depending on where the scheduler puts them
        os.sched_setaffinity(0, {cpu})
    except (AttributeError, OSError):
        pass
    from lightweight_snappy_b200 import corpus
    import oracle_lib
    data = corpus.make_corpus(kind, n_bytes, seed=SEED, first_segment=shard * (n_bytes >> 20)).numpy()
    codec = oracle_lib.Reference() if use_ref else oracle_lib.Oracle()
    t0 = time.perf_counter()
    stream = codec.compress(data, mode)
    t1 = time.perf_counter()
    back = codec.decompress(stream, data.size)
    t2 = time.perf_counter()
    ok = bool(back.size == data.size and np.array_equal(back, data))
    return {"n": int(data.size), "c": int(stream.size), "t_comp": t1 - t0, "t_decomp": t2 - t1, "ok": ok}


def cpu_baseline(sample_mib_per_core: int = 48, cores: int | None = None, kind: str = "mixed", mode: int = 0) -> dict:
    """Reference CPU codec, one pinned process per host core, each on its own shard (BASELINE.md 3).
    The sample is BOUNDED (cores x sample_mib_per_core MiB of the same corpus generator), not the
    whole 1 GiB workload: the CPU codec's throughput does not depend on the input size."""
    import multiprocessing as mp
    import oracle_lib
    if not os.path.exists(oracle_lib.ORACLE_SO):
        oracle_lib.build(ref=False)
    use_ref = oracle_lib.Reference.available()
    try:
        cpus = sorted(os.sched_getaffinity(0))
    except AttributeError:
        cpus = list(range(os.cpu_count() or 1))
    cores = min(cores or len(cpus), len(cpus))
    n = sample_mib_per_core << 20
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        res = pool.map(_cpu_worker, [(i, n, use_ref, kind, mode, cpus[i]) for i in range(cores)], chunksize=1)
    total = sum(r["n"] for r in res)
    t_d = max(r["t_decomp"] for r in res)
    t_c = max(r["t_comp"] for r in res)
    return {
        "value": total / t_d / 1e9, "unit": "GB/s", "cores": cores, "kind": "reference" if use_ref else "port",
        "sample": f"bounded sample: {cores} x {sample_mib_per_core} MiB shards of the {kind} corpus (same generator and "
                  f"seed as the GPU arm's 1 GiB), one pinned process per core, mode {'bst' if mode else 'hash'}, "
                  f"aggregate = total bytes / slowest process",
        "shard_compressed_bytes": [r["c"] for r in res], "shard_mib": sample_mib_per_core,
        "compress_value": total / t_c / 1e9,
        "single_core_decompress": res[0]["n"] / res[0]["t_decomp"] / 1e9,
        "single_core_compress": res[0]["n"] / res[0]["t_comp"] / 1e9,
        "ratio": total / sum(r["c"] for r in res), "roundtrip_ok": all(r["ok"] for r in res),
    }


# ------------------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self) -> dict:
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.count(",") >= 6]
        os.unlink(self.f.name)
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0]))
                smax.append(float(r[1]))
            except ValueError:
                continue
            for name, v in zip(names, r[3:7]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        busy = [v for v in sm if v >= 0.5 * max(smax)] if sm else []
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------ reference arm
def run_reference_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # a "step" is one bounded sample (16 x 48 MiB shards through the reference, ~10 s); W is capped
    # at 1 warm-up, K steps are timed as asked
    warm = min(max(args.warmup, 0), 1)
    for _ in range(warm):
        cpu_baseline()
    base = cpu_baseline()
    vals = [base["value"]]
    for _ in range(args.steps - 1):
        vals.append(cpu_baseline()["value"])
    v = statistics.median(vals)
    base["value"] = v
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "GB/s", "n_gpus": args.gpus, "steps": len(vals),
        "warmup": warm, "ms_per_step": None, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": "mixed corpus (text/low-entropy/random, 1 MiB segments), decompression, "
                               "reference CPU build on all host cores; BOUNDED SAMPLE of the GPU arm's 1 GiB workload "
                               "(16 x 48 MiB shards per step, same generator and seed) -- CPU throughput is "
                               "size-independent, so the config differs from the GPU arm by design",
                   "spread": {"min": min(vals), "max": max(vals), "samples": len(vals)}},
        "cpu_baseline": base,
        "e2e": {"value": v, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "compress": {"value": base["compress_value"], "unit": "GB/s"},
    }
    emit(line)


# ------------------------------------------------------------------------------ FILE* layer / CLI
def file_layer_e2e(api, data, c_bytes: int) -> dict:
    import ctypes as C
    import shutil
    d = tempfile.mkdtemp(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        src, comp, back = (os.path.join(d, x) for x in ("in.bin", "out.snp", "back.bin"))
        data.tofile(src)
        n = data.size
        libc = C.CDLL(None)
        libc.fopen.restype = C.c_void_p
        libc.fopen.argtypes = [C.c_char_p, C.c_char_p]
        libc.fclose.argtypes = [C.c_void_p]
        L = api.lib()
        L.snappy_compress.restype = None
        L.snappy_compress.argtypes = [C.c_void_p, C.c_ulonglong, C.c_void_p]
        L.snappy_decompress.restype = C.c_int
        L.snappy_decompress.argtypes = [C.c_void_p, C.c_void_p]

        def call(fn, a, b, *extra):
            fi, fo = libc.fopen(a.encode(), b"rb"), libc.fopen(b.encode(), b"wb")
            t0 = time.perf_counter()
            fn(fi, *extra, fo)
            libc.fclose(fo)
            dt = time.perf_counter() - t0
            libc.fclose(fi)
            return dt

        call(L.snappy_compress, src, comp, n)  # warm-up (page-locked buffers, module load)
        t_c = min(call(L.snappy_compress, src, comp, n) for _ in range(2))
        assert os.path.getsize(comp) == c_bytes, "FILE* layer: stream size differs"
        call(L.snappy_decompress, comp, back)
        t_d = min(call(L.snappy_decompress, comp, back) for _ in range(2))
        assert os.path.getsize(back) == n
        out = {"bytes": n, "where": "tmpfs (/dev/shm)" if d.startswith("/dev/shm") else d,
               "dropin_compress_GBs": n / t_c / 1e9, "dropin_decompress_GBs": n / t_d / 1e9,
               "dropin": "snappy_compress / snappy_decompress on FILE*, in process, warm, fclose included"}
        t0 = time.perf_counter()
        subprocess.run([api.CLI_PATH, "-c", src, comp], check=True)
        t1 = time.perf_counter()
        subprocess.run([api.CLI_PATH, "-d", comp, back], check=True)
        t2 = time.perf_counter()
        import numpy as np
        assert np.array_equal(np.fromfile(back, np.uint8), data), "CLI round trip failed"
        out.update({"cli_compress_GBs": n / (t1 - t0) / 1e9, "cli_decompress_GBs": n / (t2 - t1) / 1e9,
                    "cli": "snappy_b200 -c / -d, one process per call (CUDA start-up and page-locking included)"})
        return out
    finally:
        shutil.rmtree(d, ignore_errors=True)


# ------------------------------------------------------------------------------ --dump-outputs
def _seeded_positions(n: int, k: int):
    """k sorted positions in [0, n), a function of (SEED, n, k) only; None when n <= k (keep everything)."""
    import numpy as np
    if n <= k:
        return None
    return np.sort(np.random.default_rng(SEED).integers(0, n, size=k))


def _save_values(out_dir: str, name: str, t, k: int, dtype) -> int:
    import numpy as np
    import torch
    pos = _seeded_positions(t.numel(), k)
    if pos is not None:
        t = t[torch.from_numpy(pos).to(t.device)]
    path = os.path.join(out_dir, name + ".npy")
    np.save(path, t.cpu().numpy().astype(dtype))
    return os.path.getsize(path)


def dump_leg(out_dir: str, leg: str, data_name: str, data, offsets) -> int:
    """One timed leg's results: a uint8 device tensor (sampled bytes + 64 KiB chunk sums, so that every byte
    counts) and its block offsets.  Returns the bytes written."""
    import numpy as np
    import torch
    chunk = 1 << 16
    n = data.numel()
    full = n // chunk * chunk
    sums = data[:full].view(-1, chunk).sum(1, dtype=torch.int64)
    if full < n:
        sums = torch.cat([sums, data[full:].sum(dtype=torch.int64).view(1)])
    return (_save_values(out_dir, f"{leg}_{data_name}_sample", data, DUMP_SAMPLE, np.float32)
            + _save_values(out_dir, f"{leg}_{data_name}_chunk_sums", sums, DUMP_MAX_ENTRIES, np.float64)
            + _save_values(out_dir, f"{leg}_block_offsets", offsets, DUMP_MAX_ENTRIES, np.float64))


# ------------------------------------------------------------------------------ GPU arm
def measured_peak() -> tuple[float, str]:
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def run_gpu_arm(args) -> None:
    import torch
    import torch.distributed as dist
    from lightweight_snappy_b200 import api, corpus

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # keep stdout for the one JSON line
        dist.init_process_group("nccl", device_id=dev)

    base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        base = cpu_baseline()

    n = int(args.gib * GIB)
    seg0 = rank * (n >> 20)  # every rank owns its own slice of the corpus
    data = corpus.make_corpus("mixed", n, seed=SEED, device=dev, first_segment=seg0)
    codec = api.DeviceCodec(n, device=dev)
    out = torch.empty(n, dtype=torch.uint8, device=dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- setup: one compression gives the stream every decompression step consumes
    codec.compress(data, api.MODE_HASH)
    stream = codec.result_stream().clone()
    c_bytes = stream.numel()
    side_index = codec.block_offsets.clone()
    hdr = 1
    while (n >> (7 * hdr)) > 0:
        hdr += 1
    k0_index = torch.zeros_like(side_index)

    def step_decompress(ev=None):
        # the call a user makes for a device-resident, index-less stream: K0 (boundary discovery)
        # + block decode (a device-resident stream is decoded in one piece)
        codec.decompress(stream, c_bytes, hdr, n, out, k0_index)

    def step_decode_kernel(ev=None):
        # the two halves called separately over the whole stream, so that the dominant kernel pair
        # (k_copy_literal_blocks + k_decode_seg, one launch each over all 16384 blocks) is bracketed by its own pair of events
        codec.index(stream, c_bytes, hdr, n, k0_index)
        if ev:
            ev[0].record()
        codec.decode_segments(stream, c_bytes, hdr, n, out, k0_index)
        if ev:
            ev[1].record()

    def step_compress(ev=None):
        if ev:
            ev[0].record()
        codec.compress(data, api.MODE_HASH)
        if ev:
            ev[1].record()

    # correctness of what is about to be timed (outside the timed region)
    step_decompress()
    codec.check_status()
    assert torch.equal(out, data), "round trip failed"
    assert torch.equal(k0_index, side_index), "K0 index differs from the compressor's side index"

    def timed(step, kernel_name):
        for _ in range(args.warmup):
            step()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        launches0 = api.launch_count()
        barrier()
        t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_start.record()
        for i in range(args.steps):
            step(evs[i])
        t_end.record()
        barrier()
        clocks = None
        total_ms = t_start.elapsed_time(t_end)
        try:
            # (median of the per-step spans: a host hiccup between two launches of one step is not kernel time)
            kern_ms = statistics.median(a.elapsed_time(b) for a, b in evs)
        except (ValueError, RuntimeError):  # this step does not bracket a kernel of its own
            kern_ms = None
        return {"total_ms": max_over_ranks(total_ms), "kernel_ms": kern_ms, "clocks": clocks,
                "launches": api.launch_count() - launches0, "kernel": kernel_name}

    # clocks are sampled over the whole measured section (the timed regions themselves last
    # tens of milliseconds, less than nvidia-smi needs to start); idle samples are dropped
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        time.sleep(1.0)
    td = timed(step_decompress, DECODE_KERNEL)
    codec.check_status()
    assert torch.equal(out, data), "round trip failed (pipelined path)"
    dump_dir = args.dump_outputs if rank == 0 else None
    dumped = 0
    if dump_dir:
        os.makedirs(dump_dir, exist_ok=True)
        dumped += dump_leg(dump_dir, "decompress", "output", out, k0_index)
    tk = timed(step_decode_kernel, DECODE_KERNEL)
    codec.check_status()
    td["kernel_ms"] = tk["kernel_ms"]
    td["unpipelined_ms_per_step"] = tk["total_ms"] / args.steps
    tc = timed(step_compress, "k_parse_hash_global (+ k_emit + k_scan_sizes + k_gather)")
    codec.check_status()
    if dump_dir:
        dumped += dump_leg(dump_dir, "compress", "stream", codec.result_stream(), codec.block_offsets)

    # ---- BASELINE configs[3]: the BST (exact-key) path on 1 GiB of low-entropy + random data
    tb = None
    if not args.no_bst:
        data_b = corpus.make_corpus("lowent_random", n, seed=SEED, device=dev, first_segment=seg0)

        def step_bst(ev=None):
            if ev:
                ev[0].record()
            codec.compress(data_b, api.MODE_BST)
            if ev:
                ev[1].record()

        step_bst()
        codec.check_status()
        stream_b = codec.result_stream().clone()
        cb_bytes = stream_b.numel()
        offs_b = codec.block_offsets[: api.block_count(n) + 1].cpu().numpy()
        bst_parity = "not checked (no CPU baseline on this rank)"
        base_b = None
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            # compressed size == the reference's `-b` size, shard by shard, BEFORE anything is timed
            base_b = cpu_baseline(kind="lowent_random", mode=1)
            bps = (base_b["shard_mib"] << 20) // 65536
            vlen = 1
            while ((base_b["shard_mib"] << 20) >> (7 * vlen)) > 0:
                vlen += 1
            checked = 0
            for i, cb in enumerate(base_b["shard_compressed_bytes"]):
                if (i + 1) * bps >= len(offs_b):
                    break
                mine = int(offs_b[(i + 1) * bps]) - int(offs_b[i * bps])
                assert mine == cb - vlen, f"BST shard {i}: {mine} bytes here, {cb - vlen} from the reference's -b"
                checked += 1
            assert base_b["roundtrip_ok"]
            bst_parity = (f"compressed size equal to the reference CPU `-b` on {checked} x {base_b['shard_mib']} MiB "
                          f"shards before timing; byte identity at 1 GiB is asserted in tests/test_gpu_baseline_sizes.py")
        codec.decompress(stream_b, cb_bytes, hdr, n, out)
        codec.check_status()
        assert torch.equal(out, data_b), "BST round trip failed"
        tb = timed(step_bst, "k_parse_exact_global (+ k_emit + k_scan_sizes + k_gather)")
        codec.check_status()
        tb["c_bytes"], tb["parity"], tb["base"] = cb_bytes, bst_parity, base_b
        if dump_dir:
            dumped += dump_leg(dump_dir, "bst", "stream", codec.result_stream(), codec.block_offsets)
    assert dumped <= DUMP_LIMIT, f"--dump-outputs wrote {dumped} bytes, more than {DUMP_LIMIT}"

    # ---- end to end through the host-buffer C-ABI (pinned host memory, copies inside)
    h_stream = torch.empty(c_bytes, dtype=torch.uint8, pin_memory=True)
    h_stream.copy_(stream)
    h_data = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    h_data.copy_(data)
    h_out = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    h_comp = torch.empty(codec.comp_capacity, dtype=torch.uint8, pin_memory=True)
    torch.cuda.synchronize(dev)
    e2e_steps = args.e2e_steps or args.steps

    def e2e(fn):
        for _ in range(min(args.warmup, 2)):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            fn()
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        barrier()
        return max_over_ranks(dt)

    # the box's host<->device ceiling with all ranks copying at once (the end-to-end numbers are bounded by it:
    # profiles/r02_pcie_ceiling_8gpu.json) -- the same page-locked buffers, plain copies, best of 3
    def link_rate(fn, nbytes):
        best = None
        for _ in range(3):
            barrier()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize(dev)
            dt = max_over_ranks(time.perf_counter() - t0)
            best = dt if best is None else min(best, dt)
        return sum_over_ranks(float(nbytes)) / best / 1e9

    h2d_rate = link_rate(lambda: data.copy_(h_data, non_blocking=True), n)
    d2h_rate = link_rate(lambda: h_out.copy_(out, non_blocking=True), n)
    data.copy_(h_data)
    torch.cuda.synchronize(dev)

    got = {}

    def e2e_decomp():
        got["d"] = api.decompress_host(h_stream.numpy(), out=h_out.numpy())

    def e2e_comp():
        got["c"] = api.compress_host(h_data.numpy(), api.MODE_HASH, out=h_comp.numpy())

    dt_d = e2e(e2e_decomp)
    assert got["d"].size == n and torch.equal(h_out, h_data), "e2e round trip failed"
    dt_c = e2e(e2e_comp)
    assert got["c"].size == c_bytes and torch.equal(h_comp[:c_bytes], h_stream), "e2e stream differs"
    dt_b = None
    if tb is not None:
        h_data.copy_(data_b)
        torch.cuda.synchronize(dev)

        def e2e_bst():
            got["b"] = api.compress_host(h_data.numpy(), api.MODE_BST, out=h_comp.numpy())

        dt_b = e2e(e2e_bst)
        assert got["b"].size == tb["c_bytes"] and torch.equal(h_comp[:tb["c_bytes"]].to(dev), stream_b), "e2e BST stream differs"

    # ---- the drop-in layer end to end: tmpfs file -> file through the reference's own entry points
    # (snappy_compress / snappy_decompress on FILE*, in process, warm) and through the command line (a new
    # process per call: CUDA start-up included), wall clock
    cli = None
    if rank == 0 and world == 1 and not args.no_cli:
        cli = file_layer_e2e(api, data.cpu().numpy(), c_bytes)

    clocks = sampler.stop() if sampler else None
    td["clocks"] = tc["clocks"] = clocks

    # ---- BASELINE configs[4]: the 64 GiB batch of independent blocks, block ranges over the ranks (STRONG
    # scaling: 64 / N GiB per GPU), device-resident 4 GiB sub-batches, compress then index-less decompress,
    # 1 % of the blocks checked against the oracle, whole-batch checksum (tools/batch64.py)
    batch = None
    if not args.no_batch64:
        del h_stream, h_data, h_out, h_comp, out, data
        torch.cuda.empty_cache()
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import batch64
        batch = batch64.run(argparse.Namespace(gib=args.batch_gib, sub_gib=4.0, sample=0.01, mode=0))

    # ---- aggregate over ranks
    total_u = sum_over_ranks(float(n))
    total_c = sum_over_ranks(float(c_bytes))
    total_cb_all = sum_over_ranks(float(tb["c_bytes"])) if tb is not None else 0.0
    peak, peak_src = measured_peak()

    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f)
    except Exception:
        traffic = {}

    def roofline(t, per_launch_bytes):
        achieved = per_launch_bytes / (t["kernel_ms"] * 1e-3) / 1e9
        tr = traffic.get(t["kernel"].split()[0])
        return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": tr["dram_bytes_per_launch"] if tr and n == tr.get("bytes_per_gpu") else None,
                "traffic_source": tr.get("source") if tr else None,
                "peak_source": peak_src, "kernel": t["kernel"],
                "algorithmic_bytes_per_launch": per_launch_bytes, "kernel_ms": t["kernel_ms"]}

    if rank == 0:
        ms_d = td["total_ms"] / args.steps
        ms_c = tc["total_ms"] / args.steps
        line = {
            "metric": METRIC, "value": total_u * args.steps / (td["total_ms"] * 1e-3) / 1e9, "unit": "GB/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_d,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {
                "workload": f"{args.gib:g} GiB synthetic mixed corpus per GPU (text-like/low-entropy/random, 1 MiB "
                            f"segments), decompression of the index-less reference-format stream "
                            f"(BASELINE configs[1]); compress{{}} = hash-table compression of the same corpus "
                            f"(configs[2])",
                "bytes_per_gpu": n, "compressed_bytes_per_gpu": c_bytes, "blocks_per_gpu": api.block_count(n),
                "l2": "inputs+outputs per step (>= 1.5 GiB) are far larger than the 126 MB L2; no flush needed",
                "partitioning": f"{world} rank(s), each owns its own corpus slice; no data-path collective",
            },
            "ratio": total_u / total_c,
            "roofline": roofline(td, float(n + c_bytes)),
            "decompress_unpipelined_ms_per_step": td["unpipelined_ms_per_step"],
            "e2e": {"value": total_u * e2e_steps / dt_d / 1e9, "unit": "GB/s", "h2d_bytes_per_step": c_bytes,
                    "d2h_bytes_per_step": n, "steps": e2e_steps,
                    "api": "snappy_b200_decompress_host (pinned host buffers)",
                    "link_ceiling": {"h2d_GBs": h2d_rate, "d2h_GBs": d2h_rate,
                                     "how": "all ranks copying 1 GiB page-locked buffers at once, best of 3"},
                    # full duplex: the step cannot beat the slower of its upload and its download
                    "frac_of_link_ceiling": (total_u * e2e_steps / dt_d / 1e9) /
                                            (total_u / max(total_c / h2d_rate, total_u / d2h_rate))},
            "gpu_launches": td["launches"],
            "clocks": td["clocks"],
            "compress": {
                "value": total_u * args.steps / (tc["total_ms"] * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": ms_c,
                "roofline": roofline(tc, float(n + c_bytes)),
                "e2e": {"value": total_u * e2e_steps / dt_c / 1e9, "unit": "GB/s", "h2d_bytes_per_step": n,
                        "d2h_bytes_per_step": c_bytes, "api": "snappy_b200_compress_host (pinned host buffers)",
                        "frac_of_link_ceiling": (total_u * e2e_steps / dt_c / 1e9) /
                                                (total_u / max(total_u / h2d_rate, total_c / d2h_rate))},
                "gpu_launches": tc["launches"], "clocks": tc["clocks"],
                "parity": "stream byte-identical to the oracle is asserted in tests/ and smoke(); here the "
                          "round trip and the K0 index are asserted before timing",
            },
        }
        if tb is not None:
            total_cb = total_cb_all
            line["bst"] = {
                "workload": f"{args.gib:g} GiB per GPU, 1 MiB segments alternating low-entropy / random (BASELINE "
                            f"configs[3]), exact-key (BST) compression",
                "value": total_u * args.steps / (tb["total_ms"] * 1e-3) / 1e9, "unit": "GB/s",
                "ms_per_step": tb["total_ms"] / args.steps, "ratio": total_u / total_cb,
                "roofline": roofline(tb, float(n + tb["c_bytes"])),
                "e2e": {"value": total_u * e2e_steps / dt_b / 1e9, "unit": "GB/s", "h2d_bytes_per_step": n,
                        "d2h_bytes_per_step": tb["c_bytes"], "api": "snappy_b200_compress_host (MODE_BST)"},
                "gpu_launches": tb["launches"], "parity": tb["parity"],
            }
            if tb["base"] is not None:
                b = tb["base"]
                line["bst"]["cpu_baseline"] = {"value": b["compress_value"], "unit": "GB/s", "cores": b["cores"],
                                               "kind": b["kind"], "sample": b["sample"], "ratio": b["ratio"]}
        if cli is not None:
            line["cli_e2e"] = cli
        if batch is not None:
            batch["scaling"] = "strong"
            line["batch64"] = batch
        if base is not None:
            line["cpu_baseline"] = base
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE line on stdout."""
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    # stdout carries exactly one JSON line: whatever libraries print there (NCCL's version banner, make)
    # is sent to stderr by pointing file descriptor 1 at stderr and keeping a private handle to the real stdout
    global _REAL_STDOUT
    try:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
    except OSError:
        _REAL_STDOUT = None
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--gib", type=float, default=1.0, help="corpus size per GPU in GiB")
    ap.add_argument("--e2e-steps", type=int, default=None, help="timed steps of the host-buffer legs (default: --steps)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-bst", action="store_true", help="skip the configs[3] (BST path) leg")
    ap.add_argument("--no-cli", action="store_true", help="skip the FILE* / command-line end-to-end leg")
    ap.add_argument("--no-batch64", action="store_true", help="skip the configs[4] leg (64 GiB batch, strong scaling)")
    ap.add_argument("--batch-gib", type=float, default=64.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed device legs returned in their last step as DIR/*.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1 or (args.e2e_steps is not None and args.e2e_steps < 1):
        ap.error("--steps and --e2e-steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
