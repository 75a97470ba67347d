#!/usr/bin/env python
"""Runs bench.py under torch.profiler (CUDA activity) and writes the launch list summary: per kernel launches, total
time, share.  usage: profile_launches.py OUT.txt [bench.py arguments...]"""
import collections
import os
import runpy
import sys

import torch
from torch.profiler import ProfilerActivity, profile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
out = sys.argv[1]
sys.argv = [os.path.join(ROOT, "bench.py")] + sys.argv[2:]
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    try:
        runpy.run_path(sys.argv[0], run_name="__main__")
    except SystemExit:
        pass
agg = collections.defaultdict(lambda: [0, 0.0])
for e in prof.events():
    if e.device_type == torch.autograd.DeviceType.CUDA and not e.name.startswith("Memcpy") and not e.name.startswith("Memset"):
        agg[e.name][0] += 1
        agg[e.name][1] += e.time_range.elapsed_us()
tot = sum(v[1] for v in agg.values()) or 1.0
with open(out, "w") as f:
    f.write("%-40s %8s %12s %7s\n" % ("kernel", "launches", "total_us", "share"))
    for k, (n, us) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
        f.write("%-40s %8d %12.1f %6.1f%%\n" % (k[:40], n, us, 100.0 * us / tot))
