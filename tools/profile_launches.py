"""Launch list of a command's own kernels from torch.profiler (CUDA activity), written as a CSV that
tools/launch_list.py summarises (columns "Kernel Name" and "Metric Value", kernel time in ns).

    python tools/profile_launches.py OUT.csv [--] bench.py --no-cpu-baseline ...

The command is a Python script run in this process under the profiler.  Times are the kernels' device
durations with the profiler on; compare shares, not absolutes.
"""
import csv
import os
import re
import runpy
import sys

import torch
from torch.profiler import ProfilerActivity, profile

out_csv, argv = sys.argv[1], sys.argv[2:]
if argv and argv[0] == "--":
    argv = argv[1:]
sys.argv = argv
sys.path.insert(0, os.path.dirname(os.path.abspath(argv[0])))
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    try:
        runpy.run_path(argv[0], run_name="__main__")
    except SystemExit as e:
        if e.code not in (None, 0):
            raise
    torch.cuda.synchronize()
rows = []
for ev in prof.events():
    if ev.device_type != torch.autograd.DeviceType.CUDA:
        continue
    # "void sb200::(anonymous namespace)::k_copy_literal_blocks(const unsigned char *, ...)" -> "k_copy_literal_blocks"
    name = ev.name.replace("(anonymous namespace)::", "").replace("sb200::", "").removeprefix("void ")
    name = re.sub(r"\((?:[^()]|\([^()]*\))*\)$", "", name)
    if name.startswith("k_"):
        rows.append((name, int(round(ev.time_range.elapsed_us() * 1000))))
with open(out_csv, "w", newline="") as f:
    w = csv.writer(f, quoting=csv.QUOTE_ALL)
    w.writerow(["ID", "Kernel Name", "Metric Name", "Metric Unit", "Metric Value"])
    for i, (name, ns) in enumerate(rows):
        w.writerow([i, name, "device_time", "ns", ns])
print(f"{len(rows)} launches -> {out_csv}", file=sys.stderr)
