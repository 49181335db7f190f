#!/usr/bin/env python
"""Per-read phase times of the packed DP kernel on the bench workload, from its clock64() phase timers.

    python tools/pk_phase_timers.py [--lib LIB] [--loci 32768] [--steps 4] [--json OUT]

LIB is a build of strkit_b200/csrc/api.cu with -DPK_PHASE_TIMERS=1 (without --lib the script compiles one into a
temporary directory, which takes several minutes).  The workload is bench.py's default block: config-2 reads, the
reference windows of the same loci.  For every rows-per-lane class and both modes (read path, reference path) it prints
the SM cycles per warp iteration (one read, or two with 16 lanes per read) spent in the prologue (queue pop to the
first step), the step loops and the epilogue (combine / reference reduction), and the share of the first and the last.
Cycles are summed over warps that share an SM scheduler, so a share is a share of the warps' time, not of issue slots.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NBIN = 17
PHASES = ("prologue", "steps", "epilogue")


def build_timer_lib(out_dir: str) -> str:
    sys.path.insert(0, ROOT)
    import __graft_entry__ as ge

    lib = os.path.join(out_dir, "libstrkit_b200_timers.so")
    cmd = [os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"), *ge.NVCC_FLAGS, "-DPK_PHASE_TIMERS=1", "-o", lib,
           os.path.join(ROOT, "strkit_b200", "csrc", "api.cu")]
    print("[build]", " ".join(cmd), file=sys.stderr, flush=True)
    subprocess.check_call(cmd)
    return lib


def summarize(raw) -> list[dict]:
    """raw: 2 * 2 * NBIN * 4 counters in pk_phase_clk order -> one row per (mode, lanes, R) that ran."""
    rows = []
    for mode in range(2):
        for half in range(2):
            for R in range(NBIN):
                base = ((mode * 2 + half) * NBIN + R) * 4
                cyc, iters = raw[base:base + 3], raw[base + 3]
                if not iters:
                    continue
                tot = sum(cyc)
                rows.append({"mode": "reference" if mode else "reads", "L": 16 if half else 32, "R": R, "warp_iters": iters,
                             **{f"{p}_cyc_per_iter": c / iters for p, c in zip(PHASES, cyc)},
                             "prologue_share": cyc[0] / tot, "epilogue_share": cyc[2] / tot,
                             "per_read_share": (cyc[0] + cyc[2]) / tot, "cycles": tot})
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=None, help="a -DPK_PHASE_TIMERS=1 build (default: compile one)")
    ap.add_argument("--loci", type=int, default=32768)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--json", default=None, help="also write the rows as JSON here")
    args = ap.parse_args()
    tmp = tempfile.mkdtemp(prefix="pk_timers_")
    lib_path = os.path.abspath(args.lib) if args.lib else build_timer_lib(tmp)
    os.environ["STRKIT_B200_LIB"] = lib_path
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch

    import bench
    import strkit_b200
    from strkit_b200 import synth

    raw_lib = C.CDLL(lib_path)
    fn = raw_lib.strk_pk_phase_timers  # AttributeError: not a -DPK_PHASE_TIMERS=1 build
    fn.restype, fn.argtypes = C.c_int, [C.c_int, C.c_void_p, C.c_int]
    buf = np.zeros(2 * 2 * NBIN * 4, dtype=np.uint64)

    def read(reset: int) -> np.ndarray:
        strkit_b200._native.check(fn(0, buf.ctypes.data, reset))
        return buf.copy()

    torch.cuda.set_device(0)
    eng = strkit_b200.Engine(device=0)
    params = strkit_b200.RepeatCountParams("repalign", 50, 3, 1)
    sb = synth.generate(synth.CONFIGS[2], args.loci, seed=bench.batch_seed(0, 0), device="cuda", chunk_loci=4096)
    hb, ha = sb.to_host(pin=True, nibble=True), sb.to_host()
    del sb
    dev = eng.upload(hb)
    rb, start, ref_size, rc, anchor, _ = bench.ref_windows_of(ha, np)
    stream = torch.cuda.current_stream().cuda_stream
    eng.run(dev, params, strkit_b200.KERNEL_AUTO, stream)  # warm-up
    eng.ref_counts(rb, start, ref_size, rc, anchor)
    torch.cuda.synchronize()
    read(1)
    for _ in range(args.steps):
        eng.run(dev, params, strkit_b200.KERNEL_AUTO, stream)
        eng.ref_counts(rb, start, ref_size, rc, anchor)
    torch.cuda.synchronize()
    rows = summarize(read(1).tolist())
    eng.close()
    name = torch.cuda.get_device_name(0)
    try:
        plim = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        plim = "unknown"
    print(f"# {name}, power limit {plim}; lib {os.path.basename(lib_path)}; {args.loci} loci x {args.steps} steps")
    print(f"{'mode':9s} {'L':>2s} {'R':>2s} {'warp_iters':>10s} {'prologue':>9s} {'steps':>9s} {'epilogue':>9s} "
          f"{'pro%':>5s} {'epi%':>5s} {'sum%':>5s}  (SM cycles per warp iteration)")
    for r in rows:
        print(f"{r['mode']:9s} {r['L']:2d} {r['R']:2d} {r['warp_iters']:10d} {r['prologue_cyc_per_iter']:9.0f} "
              f"{r['steps_cyc_per_iter']:9.0f} {r['epilogue_cyc_per_iter']:9.0f} {100 * r['prologue_share']:5.1f} "
              f"{100 * r['epilogue_share']:5.1f} {100 * r['per_read_share']:5.1f}")
    for mode in ("reads", "reference"):
        sel = [r for r in rows if r["mode"] == mode]
        tot = sum(r["cycles"] for r in sel)
        if tot:
            share = sum(r["cycles"] * r["per_read_share"] for r in sel) / tot
            print(f"# {mode}: prologue + epilogue = {100 * share:.1f} % of the packed kernel's warp cycles")
    if args.json:
        with open(args.json, "w") as fh:
            json.dump({"device": name, "power_limit": plim, "lib": os.path.basename(lib_path), "rows": rows}, fh, indent=1)


if __name__ == "__main__":
    main()
