#!/usr/bin/env python
"""Kernel times per rows-per-lane class of the bench workload, from a torch.profiler trace of its own.

    python tools/pk_class_times.py [--lib LIB] [--loci 32768] [--steps 4] [--json OUT]

Runs bench.py's default block (config-2 reads, then the reference windows of the same loci) once to warm up, then
--steps times under torch.profiler with CUDA activities, and prints every kernel's launches, total and mean time.
The reference path runs on this thread here (bench.py's timed region overlaps it with the reads), but the class
launches of one pass still overlap on side streams; with CUDA_LAUNCH_BLOCKING=1 every kernel runs alone, which is the
setting for comparing builds kernel by kernel.  These are per-kernel times, not a step time.  LIB selects another
build of the library.
"""
from __future__ import annotations

import argparse
import collections
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=None)
    ap.add_argument("--loci", type=int, default=32768)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    if args.lib:
        os.environ["STRKIT_B200_LIB"] = os.path.abspath(args.lib)
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch
    from torch.profiler import ProfilerActivity, profile

    import bench
    import strkit_b200
    from strkit_b200 import synth

    torch.cuda.set_device(0)
    eng = strkit_b200.Engine(device=0)
    params = strkit_b200.RepeatCountParams("repalign", 50, 3, 1)
    sb = synth.generate(synth.CONFIGS[2], args.loci, seed=bench.batch_seed(0, 0), device="cuda", chunk_loci=4096)
    hb, ha = sb.to_host(pin=True, nibble=True), sb.to_host()
    del sb
    dev = eng.upload(hb)
    rb, start, ref_size, rc, anchor, _ = bench.ref_windows_of(ha, np)
    stream = torch.cuda.current_stream().cuda_stream

    def step():
        eng.run(dev, params, strkit_b200.KERNEL_AUTO, stream)
        eng.ref_counts(rb, start, ref_size, rc, anchor)

    step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.steps):
            step()
        torch.cuda.synchronize()
    agg = collections.defaultdict(lambda: [0, 0.0])
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            a = agg[ev.name]
            a[0] += 1
            a[1] += ev.device_time_total / 1e3  # us -> ms
    eng.close()
    rows = sorted(({"kernel": k, "launches": n, "total_ms": t, "ms_per_step": t / args.steps} for k, (n, t) in agg.items()),
                  key=lambda r: -r["total_ms"])
    tot = sum(r["total_ms"] for r in rows)
    print(f"# {torch.cuda.get_device_name(0)}; lib {os.path.basename(os.environ.get('STRKIT_B200_LIB', 'libstrkit_b200.so'))}; "
          f"{args.loci} loci x {args.steps} steps (reads + reference windows); {tot / args.steps:.3f} ms of kernels per step")
    for r in rows:
        print(f"{r['kernel'][:60]:60s} n={r['launches']:5d} ms/step={r['ms_per_step']:8.3f} share={r['total_ms'] / tot:.3f}")
    if args.json:
        with open(args.json, "w") as fh:
            json.dump({"device": torch.cuda.get_device_name(0), "steps": args.steps, "loci": args.loci, "rows": rows}, fh, indent=1)


if __name__ == "__main__":
    main()
