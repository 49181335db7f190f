#!/usr/bin/env python
"""bench.py -- throughput of the per-read repeat-count hot path on synthetic HiFi reads.

    python bench.py --gpus N --steps K --warmup W            (our CUDA path)
    python bench.py --impl reference --gpus N --steps K ...  (the reference's CPU path, host cores)
    python bench.py --steps K --dump-outputs DIR              (also writes what step K returned, for comparing builds)

A "step" is one pass of the hot path over one batch (loci_per_step loci x 30 reads, BASELINE config 2
distributions: "synthetic genome-wide catalog 1M loci x 30x HiFi reads, loci sharded across GPUs").  The
default K x loci_per_step is the full 1M-locus catalog on one GPU.  Multi-GPU: loci are sharded by catalog
partition, one rank per GPU, NO collective on the data path (weak scaling: every rank gets its own
loci_per_step per step); torch.distributed is used for the barriers and the max-over-ranks timing only.

Printed JSON (one line, rank 0): metric / value = reads x loci per second with the batch resident in HBM;
e2e = the same through the host-buffer C-ABI call (pinned host arenas, H2D + kernels + D2H inside the
timed region); roofline = the DP kernel against the measured integer issue rate; cpu_baseline = the CPU
oracle (a port of the reference's algorithm; the real parasail/strkit_rust_ext are not installable here)
timed on this box's host cores over a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "read x locus repeat counts per second"
UNIT = "reads*loci/s"
READS_PER_LOCUS = 30


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--loci-per-step", type=int, default=32768)
    ap.add_argument("--pool", type=int, default=4, help="distinct synthetic batches cycled through (> L2)")
    ap.add_argument("--kernel", default="auto", choices=["auto", "general"])
    ap.add_argument("--cpu-sample-loci", type=int, default=0,
                    help="cap on the loci per step the CPU arms run (0 = as many as the time budget allows)")
    ap.add_argument("--cpu-budget-s", type=float, default=200.0,
                    help="--impl reference: time budget of the W + K steps (full steps if they fit, else a sample of each)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-ref-path", action="store_true", help="time the read path only (round-1 definition of value)")
    ap.add_argument("--ascii-arenas", action="store_true", help="host arenas one byte per symbol instead of nibble-packed")
    ap.add_argument("--sustain-s", type=float, default=6.0, help="length of the sustained leg (0 = skip)")
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4], help="BASELINE.json config (2 = the headline)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="strong: ONE 1M-locus catalog partitioned over the ranks by DP area, results gathered on rank 0")
    ap.add_argument("--strong-sub-blocks", type=int, default=0,
                    help="--scaling strong: stream a partition in blocks of about 1/N of it (0 = the catalog's own blocks)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = the same number of blocks as --steps")
    ap.add_argument("--loci3", type=int, default=100_000, help="--config 3: loci in the config")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (rank 0: per-read counts, reference-window counts) "
                         "to DIR/<name>.npy as float64; default workload only")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.config != 2 or args.scaling != "weak"):
        ap.error("--dump-outputs: the default workload only (--impl ours --config 2 --scaling weak)")
    if args.dump_outputs and args.steps < 1:
        ap.error("--dump-outputs needs at least one timed step")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays, limit=DUMP_LIMIT_BYTES):
    """Writes every array of `arrays` (name -> 2-D array of int32 results) as out_dir/<name>.npy in float64, which
    holds each int32 exactly.  Above `limit` bytes in all, each array keeps the same share of its rows: a sample drawn
    by np.random.default_rng(0), sorted, so that it depends on the array shapes only and two builds run with the same
    arguments write the same rows."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.shape[0] * a.shape[1] * 8 for a in arrays.values())
    for name, a in arrays.items():
        if total > limit:
            keep = int(a.shape[0] * limit // total)
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, dtype=np.float64))


def workload_name(args):
    return (f"cfg2: synthetic genome-wide catalog, HiFi-like reads, motif 2-6 bp x 10-60 copies, "
            f"{READS_PER_LOCUS} reads/locus, {args.loci_per_step} loci per step per GPU "
            f"({args.steps * args.loci_per_step} loci per GPU in the timed region)")


def config_dict(args, world):
    """The workload both arms (ours, --impl reference) run and print: same generator, seeds, block size, search."""
    return {"workload": workload_name(args), "reads_per_locus": READS_PER_LOCUS,
            "loci_per_step_per_gpu": args.loci_per_step, "search": "max_iters 50, range 3, step 1",
            "alignment": "parasail sg (all ends free), match 2 / mismatch -7 / indel 5",
            "l2": f"inputs larger than L2: pool of {args.pool} distinct batches "
                  f"({args.pool * args.loci_per_step * READS_PER_LOCUS * 300 / 1e6:.0f} MB of reads per GPU), cycled",
            "parallelism": f"catalog partition x{world}, no collective"}


def batch_seed(rank, p):
    return 20261018 + 2000 + 100 * rank + p


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
                power.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def ncu_dram_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel, from the committed
    `ncu --set full` summary (profiles/, a separate run under the profiler; None if the file is not there)."""
    import re

    path = os.path.join(ROOT, "profiles", "r2_full_packed_r10.txt")
    if not os.path.exists(path):
        return None, None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    total, kernel = 0.0, None
    for line in open(path):
        if line.startswith("# kernel:"):
            if kernel is not None:
                break  # first kernel of the capture only
            kernel = line.split(":", 1)[1].strip().split("(")[0]
        m = re.match(r"dram__bytes_(read|write)\.sum\s+(\w+)\s+([0-9.]+)", line)
        if m and kernel is not None:
            total += float(m.group(3)) * unit.get(m.group(2), 1.0)
    return (total or None), f"{kernel}, one launch, profiles/r2_full_packed_r10.txt"


def cpu_baseline(batch, n_loci_sample, steps=1):
    """The oracle (port of the reference's CPU algorithm) on the first n_loci_sample loci, all host cores."""
    from tests import oracle_lib

    orc = oracle_lib.load()
    cores = os.cpu_count() or 1
    sub = batch.slice_loci(0, min(n_loci_sample, batch.n_loci))
    best, cells = None, 0.0
    for _ in range(max(1, steps)):
        t0 = time.perf_counter()
        out, cells = orc.count_loci(sub.arena, sub.seq_off, sub.lens, sub.est_cn, sub.read_begin, sub.motif_off,
                                    sub.motif_len, n_threads=cores)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return {"value": sub.n_reads / best, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"first {sub.n_loci} loci ({sub.n_reads} reads) of batch 0, {best:.2f} s, "
                      f"{cells / best / 1e9:.2f} GCUPS reference-equivalent",
            "gcups": cells / best / 1e9}, out, sub


def _import_synth_without_native():
    """strkit_b200.synth (the generator both arms share) WITHOUT running the package's __init__, which loads the CUDA
    library: the reference arm must not touch the product.  A bare namespace stands in for the package; synth and
    batcher are pure Python (torch / numpy only); the C packing helper is kept out as well."""
    import types

    if "strkit_b200" in sys.modules:
        raise RuntimeError("the reference arm must start from a process that has not imported strkit_b200")
    pkg = types.ModuleType("strkit_b200")
    pkg.__path__ = [os.path.join(ROOT, "strkit_b200")]
    sys.modules["strkit_b200"] = pkg
    sys.modules["strkit_b200._fastpack"] = None  # ImportError inside batcher -> its pure-Python body
    from strkit_b200 import synth

    assert "strkit_b200._native" not in sys.modules and "strkit_b200.engine" not in sys.modules
    return synth


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores, same config / metric / unit.
    parasail and strkit_rust_ext cannot be installed here or on the GPU box (profiles/r2_probe_*.txt), so this is the
    oracle port with its alignments routed through the AVX2 scan kernel (16-bit lanes, striped profile: the layout of
    the parasail kernels the reference calls; bit-identical to the scalar restatement), one thread per host core,
    the reference's lru_cache kept as a per-locus memo.  Nothing of strkit_b200's native code is loaded."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch  # noqa: F401  (data synthesis only)

    t_all = time.perf_counter()
    synth = _import_synth_without_native()
    from tests import oracle_lib

    orc = oracle_lib.load()
    simd = orc.have_simd()
    orc.set_simd(True)
    cores = os.cpu_count() or 1
    steps, warm = max(1, args.steps), max(0, args.warmup)
    # A probe gives this host's rate.  If W + K full steps (loci_per_step loci each, the very batches rank 0 of our arm
    # runs) fit the time budget they are run as they are; otherwise every step is the first n loci of its batch.
    probe = synth.generate(synth.CONFIGS[2], 1024, seed=20261018 + 1999, device="cpu").to_host()
    t0 = time.perf_counter()
    orc.count_loci(probe.arena, probe.seq_off, probe.lens, probe.est_cn, probe.read_begin, probe.motif_off,
                   probe.motif_len, n_threads=cores)
    loci_per_s = probe.n_loci / (time.perf_counter() - t0)
    budget_s = float(args.cpu_budget_s)
    n_sample = int(min(args.loci_per_step, max(32, budget_s * loci_per_s / (steps + warm))))
    if args.cpu_sample_loci:
        n_sample = min(n_sample, args.cpu_sample_loci)
    full = n_sample == args.loci_per_step
    # CPU generation of a 32 768-locus batch takes ~50 s: full steps reuse ONE batch (nothing here fits a CPU cache
    # either way: 300 MB), sampled steps generate only the loci they time (the generator is sequential in 4096-locus
    # chunks, so these are the first loci of the batches the same seeds give at full size)
    pool = 1 if full else max(1, min(args.pool, steps))
    batches = []
    for p in range(pool):
        n_gen = args.loci_per_step if full else min(args.loci_per_step, -(-n_sample // 4096) * 4096)
        b = synth.generate(synth.CONFIGS[2], n_gen, seed=batch_seed(0, p), device="cpu", chunk_loci=4096).to_host()
        batches.append(b if full else b.slice_loci(0, n_sample, compact=True))
    times, cells, n_reads = [], 0.0, 0
    for it in range(warm + steps):
        batch = batches[it % pool]
        t0 = time.perf_counter()
        _, c = orc.count_loci(batch.arena, batch.seq_off, batch.lens, batch.est_cn, batch.read_begin,
                              batch.motif_off, batch.motif_len, n_threads=cores)
        if it >= warm:
            times.append(time.perf_counter() - t0)
            cells += c
            n_reads += batch.n_reads
    total = sum(times)
    value = n_reads / total
    sample = (f"full steps: {args.loci_per_step} loci x {READS_PER_LOCUS} reads (one batch, reused every step)" if full else
              f"first {n_sample} loci ({n_sample * READS_PER_LOCUS} reads) of each {args.loci_per_step}-locus step "
              f"(time budget {budget_s:.0f} s for {warm} + {steps} steps at {loci_per_s:.0f} loci/s)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": total / steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int16 (AVX2), int32 where 16 bits do not hold" if simd else "int32",
            "data": "synthetic", "config": config_dict(args, args.gpus),
            "gcups_reference_equivalent": cells / total / 1e9,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "simd": "avx2 int16" if simd else None,
                             "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "native_modules_loaded": sorted(m for m in sys.modules if m.startswith("strkit_b200.") and sys.modules[m] is not None),
            "wall_s": time.perf_counter() - t_all}
    print(json.dumps(line), flush=True)


def run_other_config(args):
    """--config 3 / 4: the other read-path configs of BASELINE.json through the same calls (single GPU): resident
    timing with CUDA events, the streamed host-buffer path, roofline of the DP kernels, CPU port on a bounded sample."""
    import numpy as np
    import torch

    import strkit_b200
    from strkit_b200 import synth
    from tests import oracle_lib

    if int(os.environ.get("WORLD_SIZE", "1")) != 1:
        raise SystemExit("--config 3 / 4 run on one GPU")
    torch.cuda.set_device(0)
    eng = strkit_b200.Engine(device=0)
    params = strkit_b200.RepeatCountParams("repalign", 50, 3, 1)
    if args.config == 3:
        n_loci, block = args.loci3, 16384
        name = f"cfg3: {n_loci} loci x 40 ONT-like reads (~5% errors, indel-dominated), blocks of {block} loci"
        batches = [synth.generate(synth.CONFIGS[3], min(block, n_loci - lo), seed=20261018 + 3000 + i, device="cuda")
                   .to_host(pin=True, nibble=not args.ascii_arenas) for i, lo in enumerate(range(0, n_loci, block))]
    else:
        name = ("cfg4: 60 loci x 50 reads, the 44 motifs of catalogs/pathogenic_assoc.hg38.tsv (+16 resampled), one allele "
                "10-40 copies, the other 200-2000 copies capped at a 6 kb tract")
        batches = [synth.generate_expansions(60, 50)[0]]
    dev_batches = [eng.upload(b) for b in batches]
    stream = torch.cuda.current_stream().cuda_stream
    peak = eng.measure_int_peak()
    STAT_KEYS = ("executed_cells", "reference_cells", "kernel_launches", "dp_ms", "replay_ms", "widening_passes",
                 "reads_packed_kernel", "reads_general_kernel")
    for w in range(args.warmup):
        for db in dev_batches:
            eng.run(db, params, 0, stream)
    sampler = ClockSampler(0)
    sampler.start()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    agg = {k: 0.0 for k in STAT_KEYS}
    ev0.record()
    for k in range(args.steps):   # a step = one pass over the whole config
        for db in dev_batches:
            eng.run(db, params, 0, stream)
            st = eng.stats()
            for key in agg:
                agg[key] += st[key]
    ev1.record()
    torch.cuda.synchronize()
    elapsed_ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop()
    reads = sum(b.n_reads for b in batches)
    outs = [np.empty((b.n_reads, 4), dtype=np.int32) for b in batches]
    for _ in eng.count_reads_stream(batches[:2], params, outs=outs[:2]):
        pass
    t0 = time.perf_counter()
    for k in range(args.steps):
        for _ in eng.count_reads_stream(batches, params, outs=outs):
            pass
    dt_e2e = time.perf_counter() - t0
    orc = oracle_lib.load()
    orc.set_simd(True)
    cores = os.cpu_count() or 1
    b0 = batches[0].to_ascii()
    sub = b0.slice_loci(0, min(b0.n_loci, args.cpu_sample_loci or (2048 if args.config == 3 else 6)), compact=True)
    t0 = time.perf_counter()
    want, cells = orc.count_loci(sub.arena, sub.seq_off, sub.lens, sub.est_cn, sub.read_begin, sub.motif_off, sub.motif_len,
                                 n_threads=cores)
    dt_cpu = time.perf_counter() - t0
    parity = bool(np.array_equal(outs[0][:sub.n_reads], want))
    dp_s = agg["dp_ms"] * 1e-3
    achieved = agg["executed_cells"] * 4.0 / dp_s / 1e12 if dp_s > 0 else 0.0
    steps = max(1, args.steps)
    line = {"metric": METRIC, "value": reads * steps / (elapsed_ms * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": elapsed_ms / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u16x2/int32", "data": "synthetic",
            "config": {"workload": name, "reads_per_step": reads, "search": "max_iters 50, range 3, step 1",
                       "l2": f"inputs larger than L2: {sum(b.nbytes() for b in batches) / 1e6:.0f} MB per pass"
                             if args.config == 3 else "inputs smaller than L2 (6 MB): the config is 3 000 reads"},
            "gcups_executed": agg["executed_cells"] / (elapsed_ms * 1e-3) / 1e9,
            "gcups_reference_equivalent": agg["reference_cells"] / (elapsed_ms * 1e-3) / 1e9,
            "roofline": {"bound": "int_alu", "achieved": achieved, "peak": peak["dual_pipe"], "unit": "Tiop/s",
                         "frac": achieved / peak["dual_pipe"], "traffic": None, "ops_per_cell": 4,
                         "kernel": "dp_packed_kernel + dp_general_kernel" if agg["reads_packed_kernel"] else "dp_general_kernel",
                         "kernel_ms_per_step": agg["dp_ms"] / steps, "kernel_share_of_step": agg["dp_ms"] / elapsed_ms},
            "e2e": {"value": reads * steps / dt_e2e, "unit": UNIT, "h2d_bytes_per_step": int(sum(b.nbytes() for b in batches)),
                    "d2h_bytes_per_step": int(sum(o.nbytes for o in outs)), "how": "Engine.count_reads_stream over the blocks"},
            "cpu_baseline": {"value": sub.n_reads / dt_cpu, "unit": UNIT, "cores": cores, "kind": "port", "simd": "avx2 int16",
                             "sample": f"first {sub.n_loci} loci ({sub.n_reads} reads), {dt_cpu:.2f} s",
                             "gcups": cells / dt_cpu / 1e9},
            "gpu_launches": int(agg["kernel_launches"]), "widening_passes": int(agg["widening_passes"]),
            "reads_packed_kernel": int(agg["reads_packed_kernel"]), "reads_general_kernel": int(agg["reads_general_kernel"]),
            "parity_sample_bit_exact": parity, "clocks": clocks}
    print(json.dumps(line), flush=True)


def strong_scaling_line(args, world, n_blocks, block, total_reads, t_total, per_rank, loci_per_rank, sub_block, h2d_per_block,
                        d2h_per_block, launches, parity_ok, clocks, numa_note):
    """The JSON line of --scaling strong (plain numbers in, a json.dumps-able dict out: tested on the CPU)."""
    cfg = config_dict(args, world)
    cfg["parallelism"] = (f"ONE catalog of {n_blocks * block} loci cut into {world} contiguous partitions of equal "
                          "estimated DP area; no collective on the data path, one gather of the results to rank 0")
    cfg["host_affinity"] = numa_note
    per_rank = [float(t) for t in per_rank]
    return {"metric": METRIC, "value": total_reads / t_total, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t_total / n_blocks * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u16x2/int32", "data": "synthetic", "config": cfg,
            "value_is": "whole job, host buffers in -> gathered host results out (reads + reference windows)",
            "e2e": {"value": total_reads / t_total, "unit": UNIT, "h2d_bytes_per_step": int(h2d_per_block),
                    "d2h_bytes_per_step": int(d2h_per_block)},
            "partition": {"loci_per_rank": [int(x) for x in loci_per_rank], "loci_per_streamed_block": int(sub_block),
                          "compute_s_per_rank": per_rank, "imbalance_max_over_mean": max(per_rank) / (sum(per_rank) / world),
                          "gather_s": t_total - max(per_rank), "total_s": t_total,
                          "gather": "per-block D2H straight into one shared-memory result array; closing barrier"},
            "gpu_launches": int(launches), "parity_sample_bit_exact": bool(parity_ok), "clocks": clocks}


def run_strong_scaling(args, world, rank, local_rank, dev, barrier, reduce_max, numa_note):
    """--scaling strong: ONE catalog of steps x loci_per_step loci (default 32 x 32 768 = 1M loci x 30 reads), cut into
    `world` contiguous partitions of equal estimated DP area (sharding.partition_catalog); every rank streams its
    partition through the host-buffer path (reads + reference windows) and the per-read results are gathered on rank 0
    in catalog order -- inside the timed region -- where the reference heap-merges its workers' results
    (call_sample.py:420).  No collective on the data path: the one gather moves 16 bytes per read."""
    import numpy as np
    import torch
    import torch.distributed as dist

    import strkit_b200
    from strkit_b200 import sharding, synth

    n_blocks, block = max(1, args.steps), args.loci_per_step
    eng = strkit_b200.Engine(device=local_rank)
    params = strkit_b200.RepeatCountParams("repalign", 50, 3, 1)
    register = lambda a: strkit_b200._native.check(strkit_b200._native.lib.strk_host_register(a.ctypes.data, a.nbytes))  # noqa: E731
    # pass 1 (every rank, same seeds -> same catalog): per-locus cost of the whole catalog
    costs, reads_per_block = [], []
    for i in range(n_blocks):
        sb_ = synth.generate(synth.CONFIGS[2], block, seed=batch_seed(0, i), device=str(dev), chunk_loci=4096)
        n1 = sb_.lens.sum(dim=1).double()
        per_read = n1 * n1
        csum = torch.cat([per_read.new_zeros(1), per_read.cumsum(0)])
        costs.append((csum[sb_.read_begin[1:]] - csum[sb_.read_begin[:-1]]).cpu().numpy())
        reads_per_block.append(int(sb_.est_cn.numel()))
        del sb_
    cost = np.concatenate(costs)
    bounds = sharding.partition_catalog(cost, world)
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    # pass 2: the blocks of my partition, as host arrays (nibble-packed, pinned) + their reference windows
    # The partition is streamed in the catalog's own blocks (32 768 loci).  --strong-sub-blocks K: blocks of about 1 / K
    # of the partition instead -- the first block's copy and the last block's download are the part of the stream that
    # nothing overlaps, so smaller blocks should help a rank with a small partition.  Measured with K = 12: N = 4
    # unchanged (213.4 M), N = 8 202.7 M with ONE rank at 155 ms and seven at 71-76 ms (whole blocks: 397.4 M, every rank
    # at 74-78 ms); not re-measured, so the proven layout stays the default.
    sub_block = block
    if args.strong_sub_blocks > 0:
        sub_block = int(min(block, max(4096, -(-((hi - lo) // args.strong_sub_blocks) // 1024) * 1024)))
    mine, refs = [], []
    for i in range(n_blocks):
        b_lo, b_hi = max(lo, i * block), min(hi, (i + 1) * block)
        if b_hi <= b_lo:
            continue
        sb_ = synth.generate(synth.CONFIGS[2], block, seed=batch_seed(0, i), device=str(dev), chunk_loci=4096)
        whole = sb_.to_host()
        del sb_
        for s0 in range(b_lo, b_hi, sub_block):
            ha = whole.slice_loci(s0 - i * block, min(s0 + sub_block, b_hi) - i * block, compact=True)
            hb = ha.to_nibble()
            for a in (hb.arena, hb.seq_off, hb.lens, hb.est_cn, hb.read_begin, hb.motif_off, hb.motif_len):
                register(a)
            mine.append(hb)
            ref = ref_windows_of(ha, np)
            for a in (ref[0].arena, ref[0].seq_off, ref[0].lens, ref[0].motif_off, ref[0].motif_len, ref[1], ref[2], ref[3], ref[5]):
                register(a)
            refs.append(ref)
    torch.cuda.empty_cache()
    n_mine = sum(b.n_reads for b in mine)
    # read counts per rank (every rank can compute them: reads per locus is constant in this catalog)
    counts = [int((bounds[r + 1] - bounds[r]) * READS_PER_LOCUS) for r in range(world)]
    assert counts[rank] == n_mine
    # The host-side gather (where the reference heap-merges its workers' results, call_sample.py:420): ONE result array
    # [total reads, 4] in catalog order lives in POSIX shared memory; every rank's per-block downloads (D2H) land
    # directly in its slice of it, so after the closing barrier rank 0 holds the whole catalog's results without
    # another copy.  (sharding.count_reads_sharded is the torch.distributed form of the same gather, for callers
    # without a shared address space.)
    from multiprocessing import shared_memory

    total_reads = n_blocks * block * READS_PER_LOCUS
    shm_name = f"strk_b200_{os.environ.get('MASTER_PORT', '0')}_{os.getppid() if world > 1 else os.getpid()}"
    shm = None
    if rank == 0:
        try:
            shared_memory.SharedMemory(name=shm_name).unlink()
        except FileNotFoundError:
            pass
        shm = shared_memory.SharedMemory(name=shm_name, create=True, size=total_reads * 16)
    barrier()
    if rank != 0:
        shm = shared_memory.SharedMemory(name=shm_name)
    result = np.ndarray((total_reads, 4), dtype=np.int32, buffer=shm.buf)
    outs, at = [], sum(counts[:rank])
    for b_ in mine:
        outs.append(result[at:at + b_.n_reads])
        at += b_.n_reads
    for o in outs:
        register(o)
    # warm both contexts and grow their recycled device buffers to the LARGEST block of the partition (a partition
    # that starts inside a block begins with a short one: growing the buffers later would put cudaMalloc / cudaFree,
    # which synchronise the device, inside the timed region)
    big = max(range(len(mine)), key=lambda i: (mine[i].n_reads, mine[i].arena.nbytes)) if mine else 0
    for w in range(max(1, args.warmup)):
        for _ in eng.count_reads_stream([mine[big], mine[big]], params, outs=[outs[big], outs[big]], refs=[refs[big], refs[big]]):
            pass
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    launches0 = eng.total_launches
    t0 = time.perf_counter()
    for _ in eng.count_reads_stream(mine, params, outs=outs, refs=refs):
        pass
    torch.cuda.synchronize()
    t_compute = time.perf_counter() - t0
    barrier()                                # every rank's rows are in the shared array: the gather is complete
    t_total = time.perf_counter() - t0
    clocks = sampler.stop()
    t_total = reduce_max(t_total)
    per_rank = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
    if world > 1:
        dist.all_gather(per_rank, torch.tensor([t_compute], dtype=torch.float64, device=dev))
        per_rank = [float(t.item()) for t in per_rank]
    else:
        per_rank = [t_compute]
    if rank == 0:
        assert result.shape[0] == total_reads
        # spot check of rows that came from the LAST rank's partition (and of rank 0's own) against the CPU port
        from tests import oracle_lib

        orc = oracle_lib.load()
        orc.set_simd(True)
        ok = True
        for locus0 in (int(bounds[world - 1]), 0):
            i = locus0 // block
            sb_ = synth.generate(synth.CONFIGS[2], block, seed=batch_seed(0, i), device=str(dev), chunk_loci=4096)
            sub = sb_.to_host().slice_loci(locus0 - i * block, min(block, locus0 - i * block + 64), compact=True)
            del sb_
            want, _ = orc.count_loci(sub.arena, sub.seq_off, sub.lens, sub.est_cn, sub.read_begin, sub.motif_off,
                                     sub.motif_len, n_threads=os.cpu_count() or 1)
            r0 = locus0 * READS_PER_LOCUS
            ok = ok and bool(np.array_equal(result[r0:r0 + sub.n_reads], want))
        line = strong_scaling_line(args, world, n_blocks, block, total_reads, t_total, per_rank,
                                   [int(bounds[r + 1] - bounds[r]) for r in range(world)], sub_block,
                                   int(sum(b.nbytes() for b in mine) / max(1, len(mine))),
                                   int(sum(o.nbytes for o in outs) / max(1, len(outs))),
                                   int(eng.total_launches - launches0), ok, clocks, numa_note)
        print(json.dumps(line), flush=True)
    for o in outs:
        strkit_b200._native.lib.strk_host_unregister(o.ctypes.data)
    del result, outs
    barrier()
    shm.close()
    if rank == 0:
        shm.unlink()


def ref_windows_of(hb, np):
    """The reference-genome window of every locus of a read batch (one sequence per locus: its first read stands in for
    the reference, error channel included) as the arrays strk_ref_counts takes (get_ref_repeat_count, repeats.py:73-192;
    search tier of < 200 copies: 250 iterations, range 3, step 1, repeat_count_params.py:25-27; vcf_anchor_size 5)."""
    from strkit_b200.batcher import ReadBatch

    first = hb.read_begin[:-1]
    lens = hb.lens[first].copy()
    tot = lens.sum(axis=1).astype(np.int64)
    r_off = np.concatenate([[0], np.cumsum(tot)[:-1]]).astype(np.int64)
    src = np.repeat(hb.seq_off[first].astype(np.int64) - r_off, tot) + np.arange(int(tot.sum()))
    ml = hb.motif_len.astype(np.int64)
    m_off = int(tot.sum()) + np.concatenate([[0], np.cumsum(ml)[:-1]]).astype(np.int64)
    msrc = np.repeat(hb.motif_off.astype(np.int64) - m_off, ml) + int(tot.sum()) + np.arange(int(ml.sum()))
    ref = ReadBatch(arena=np.concatenate([hb.arena[src], hb.arena[msrc]]), seq_off=r_off.astype(np.uint64), lens=lens,
                    est_cn=hb.est_cn[first].copy(), read_begin=np.arange(hb.n_loci + 1, dtype=np.int64),
                    motif_off=m_off.astype(np.uint64), motif_len=hb.motif_len.copy())
    rc = np.tile(np.array([250, 3, 1], dtype=np.int32), (hb.n_loci, 1))
    return (ref, ref.est_cn.copy(), ref.lens[:, 1].copy(), rc, 5, np.empty((hb.n_loci, 8), dtype=np.int32))


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    if args.config != 2:
        run_other_config(args)
        return

    import numpy as np
    import torch

    import strkit_b200
    from strkit_b200 import synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # stdout carries exactly one JSON line: keep NCCL's "NCCL version ..." banner off it (the image exports
        # NCCL_DEBUG=VERSION, and NCCL prints the banner to stdout at VERSION and at WARN)
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
            del os.environ["NCCL_DEBUG"]
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # Multi-rank runs: keep each rank's host threads and pinned arenas on the cores / memory next to its GPU.
    # Undone before the CPU baseline.
    full_affinity = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    numa_note = None
    if world > 1 and full_affinity is not None:
        try:
            import pynvml

            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
            words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
            cpus = {64 * i + b for i, wd in enumerate(words) for b in range(64) if (wd >> b) & 1} & full_affinity
            if cpus:
                os.sched_setaffinity(0, cpus)
                numa_note = f"rank pinned to the {len(cpus)} host cores local to its GPU"
        except Exception as exc:  # affinity is an optimisation, never a requirement
            numa_note = f"no GPU-local affinity ({type(exc).__name__})"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def reduce_sum(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    if args.scaling == "strong":
        run_strong_scaling(args, world, rank, local_rank, dev, barrier, reduce_max, numa_note)
        if world > 1:
            dist.destroy_process_group()
        return

    eng = strkit_b200.Engine(device=local_rank)
    params = strkit_b200.RepeatCountParams("repalign", 50, 3, 1)  # read-path defaults (params.py:45,157-163)
    kernel = strkit_b200.KERNEL_GENERAL if args.kernel == "general" else strkit_b200.KERNEL_AUTO
    register = lambda a: strkit_b200._native.check(strkit_b200._native.lib.strk_host_register(a.ctypes.data, a.nbytes))  # noqa: E731

    # ---- synthetic catalog partition of this rank: `pool` distinct batches, generated on the GPU.  Host side: the
    # batcher's nibble-packed arenas in pinned memory (what pack_loci(nibble=True) emits) + the reference window of
    # every locus; device side: the same batches resident in HBM.
    host_batches, dev_batches, ref_sets = [], [], []
    ascii0 = None
    for p in range(args.pool):
        sbatch = synth.generate(synth.CONFIGS[2], args.loci_per_step, seed=batch_seed(rank, p), device=str(dev), chunk_loci=4096)
        hb = sbatch.to_host(pin=True, nibble=not args.ascii_arenas)
        ha = sbatch.to_host() if (p == 0 or not args.no_ref_path) else None
        del sbatch
        if p == 0:
            ascii0 = ha
        host_batches.append(hb)
        dev_batches.append(eng.upload(hb))
        if not args.no_ref_path:
            ref = ref_windows_of(ha, np)
            for a in (ref[0].arena, ref[0].seq_off, ref[0].lens, ref[0].motif_off, ref[0].motif_len, ref[1], ref[2], ref[3], ref[5]):
                register(a)
            ref_sets.append(ref)
    torch.cuda.empty_cache()
    reads_per_step = host_batches[0].n_reads
    pool_bytes = sum(b.nbytes() for b in host_batches)
    stream = torch.cuda.current_stream().cuda_stream
    STAT_KEYS = ("executed_cells", "reference_cells", "kernel_launches", "dp_ms", "replay_ms", "widening_passes",
                 "reads_packed_kernel", "reads_general_kernel")

    def ref_step(k):
        rb, start, ref_size, rc, anchor, out = ref_sets[k % args.pool]
        return eng.ref_counts(rb, start, ref_size, rc, anchor)

    def ref_step_async(k):   # on the GPU's second context, under the read kernels of the same block
        rb, start, ref_size, rc, anchor, out = ref_sets[k % args.pool]
        return eng.ref_counts_async(rb, start, ref_size, rc, anchor)

    # ---- integer issue-rate peak (roofline denominator), measured on this GPU now
    peak = eng.measure_int_peak()

    # ---- warm-up (W steps of the whole hot path)
    for w in range(args.warmup):
        fut = ref_step_async(w) if ref_sets else None
        eng.run(dev_batches[w % args.pool], params, kernel, stream)
        if fut:
            fut.result()

    # ---- timed region 1 (headline `value`): K steps of the WHOLE hot path of a block of loci -- the once-per-locus
    # reference path (get_ref_repeat_count) + the per-read path -- read batches resident in HBM
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    agg = {k: 0.0 for k in STAT_KEYS}
    agg_ref = {k: 0.0 for k in STAT_KEYS}
    ref_out = None
    ev0.record()
    for k in range(args.steps):
        fut = ref_step_async(k) if ref_sets else None
        eng.run(dev_batches[k % args.pool], params, kernel, stream)
        st = eng.stats()
        for key in agg:
            agg[key] += st[key]
        if fut:
            ref_out, st = fut.result()
            for key in agg_ref:
                agg_ref[key] += st[key]
    ev1.record()
    barrier()
    elapsed_ms = reduce_max(ev0.elapsed_time(ev1))
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        # the last step's batch still holds its results on the device: download them outside the timed region
        outputs = {"read_counts": eng.download(dev_batches[(args.steps - 1) % args.pool])}
        if ref_out is not None:
            outputs["ref_counts"] = ref_out
        dump_outputs(args.dump_outputs, outputs)
    total_reads = reduce_sum(float(reads_per_step) * args.steps)
    value = total_reads / (elapsed_ms * 1e-3)
    exec_cells = reduce_sum(agg["executed_cells"] + agg_ref["executed_cells"])
    ref_cells = reduce_sum(agg["reference_cells"])

    # ---- timed region 2: the read path alone (what round 1 reported as `value`), same K steps
    barrier()
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    agg2 = {k: 0.0 for k in STAT_KEYS}   # kernel times of the read path when it has the GPU to itself: the roofline's
    ev2.record()
    for k in range(args.steps):
        eng.run(dev_batches[k % args.pool], params, kernel, stream)
        st = eng.stats()
        for key in agg2:
            agg2[key] += st[key]
    ev3.record()
    barrier()
    reads_only_ms = reduce_max(ev2.elapsed_time(ev3))

    # ---- the reference path alone (its own kernel times and roofline: in region 1 it shares the GPU with the read kernels)
    ref_solo = {k: 0.0 for k in STAT_KEYS}
    ref_solo_ms = 0.0
    if ref_sets:
        ref_step(0)   # (this context's reference-path buffers: region 1 ran the windows on the second context)
        barrier()
        t0 = time.perf_counter()
        for k in range(4):
            ref_step(k)
            st = eng.stats()
            for key in ref_solo:
                ref_solo[key] += st[key] / 4
        ref_solo_ms = (time.perf_counter() - t0) / 4 * 1e3

    # ---- sustained leg: the read path over the pool for >= --sustain-s seconds, with its own clock record
    sustained = None
    if args.sustain_s > 0:
        n_rep = max(args.steps, int(args.sustain_s * 1e3 / max(reads_only_ms / max(1, args.steps), 1e-3)) + 1)
        s2 = ClockSampler(local_rank)
        s2.start()
        barrier()
        ev4, ev5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev4.record()
        for k in range(n_rep):
            eng.run(dev_batches[k % args.pool], params, kernel, stream)
        ev5.record()
        barrier()
        sus_ms = reduce_max(ev4.elapsed_time(ev5))
        sustained = {"value": reduce_sum(float(reads_per_step) * n_rep) / (sus_ms * 1e-3), "unit": UNIT, "steps": n_rep,
                     "seconds": sus_ms * 1e-3, "what": "read path, batches resident in HBM", "clocks": s2.stop()}

    # ---- e2e: host buffers through the C-ABI calls (H2D + kernels + D2H inside the timed region), whole hot path
    e2e = None
    if not args.no_e2e:
        e2e_steps = args.e2e_steps or args.steps
        outs = [np.empty((b.n_reads, 4), dtype=np.int32) for b in host_batches]
        for o in outs:
            register(o)
        refs_of = (lambda n: (ref_sets[k % args.pool] for k in range(n))) if ref_sets else (lambda n: None)
        # (a) one blocking C-ABI call per block; (b) the streamed form: the same calls from two host threads /
        # two native contexts, the H2D copy of block i+1 overlapping the kernels of block i
        eng.count_reads(host_batches[0], params, kernel, out=outs[0])  # warm the recycled device buffers
        barrier()
        t0 = time.perf_counter()
        for k in range(e2e_steps):
            if ref_sets:
                ref_step(k)
            eng.count_reads(host_batches[k % args.pool], params, kernel, out=outs[k % args.pool])
        torch.cuda.synchronize()
        dt_call = time.perf_counter() - t0
        barrier()
        dt_call = reduce_max(dt_call)
        for _ in eng.count_reads_stream(host_batches[:2], params, kernel, outs=outs[:2], refs=refs_of(2)):  # warm both contexts
            pass
        barrier()
        t0 = time.perf_counter()
        n_done = 0
        for _ in eng.count_reads_stream((host_batches[k % args.pool] for k in range(e2e_steps)), params, kernel,
                                        outs=(outs[k % args.pool] for k in range(e2e_steps)), refs=refs_of(e2e_steps)):
            n_done += 1
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        barrier()
        dt = reduce_max(dt)
        assert n_done == e2e_steps
        # the same blocks, reads only (no reference windows): what the round-1 e2e figure measured
        t0 = time.perf_counter()
        for _ in eng.count_reads_stream((host_batches[k % args.pool] for k in range(e2e_steps)), params, kernel,
                                        outs=(outs[k % args.pool] for k in range(e2e_steps))):
            pass
        torch.cuda.synchronize()
        dt_reads = reduce_max(time.perf_counter() - t0)
        barrier()
        e2e_parity = bool(np.array_equal(outs[(e2e_steps - 1) % args.pool],
                                         eng.download(dev_batches[(e2e_steps - 1) % args.pool])))
        ref_h2d = int(sum(a.nbytes for a in (ref_sets[0][0].arena, ref_sets[0][0].seq_off, ref_sets[0][0].lens,
                                             ref_sets[0][0].motif_off, ref_sets[0][0].motif_len, ref_sets[0][1],
                                             ref_sets[0][2], ref_sets[0][3]))) if ref_sets else 0
        e2e = {"value": reduce_sum(float(reads_per_step) * e2e_steps) / dt, "unit": UNIT,
               "h2d_bytes_per_step": int(host_batches[0].nbytes()) + ref_h2d,
               "d2h_bytes_per_step": int(outs[0].nbytes) + (int(ref_sets[0][5].nbytes) if ref_sets else 0),
               "steps": e2e_steps, "ms_per_step": dt / e2e_steps * 1e3,
               "how": "Engine.count_reads_stream(refs=...): per block of loci, pinned host arrays (nibble-packed read "
                      "arena as the batcher emits it) -> strk_batch_fill_fmt / strk_ref_counts + strk_batch_run / "
                      "strk_batch_download, two host threads, copies overlapped with the kernels",
               "includes_ref_path": bool(ref_sets), "arena_format": "ascii" if args.ascii_arenas else "nibble",
               "reads_only_value": reduce_sum(float(reads_per_step) * e2e_steps) / dt_reads,
               "blocking_call_value": reduce_sum(float(reads_per_step) * e2e_steps) / dt_call,
               "equals_resident_results": e2e_parity}

    # ---- parity + CPU baseline on a bounded sample (rank 0): the first loci of batch 0 through the CPU port (AVX2
    # alignments, one thread per core), compared row by row with the device results
    cpu = None
    parity = None
    ref_parity = None
    if full_affinity is not None:
        os.sched_setaffinity(0, full_affinity)
    if rank == 0 and not args.no_cpu_baseline:
        from tests import oracle_lib

        orc = oracle_lib.load()
        orc.set_simd(True)
        cores = os.cpu_count() or 1
        n_sample = args.cpu_sample_loci or args.loci_per_step
        if world > 1:
            n_sample = min(n_sample, 1024)  # the timed CPU baseline belongs to the N = 1 line
        sub = ascii0.slice_loci(0, min(n_sample, ascii0.n_loci), compact=True)
        t0 = time.perf_counter()
        want, cells = orc.count_loci(sub.arena, sub.seq_off, sub.lens, sub.est_cn, sub.read_begin, sub.motif_off,
                                     sub.motif_len, n_threads=cores)
        dt_cpu = time.perf_counter() - t0
        if world == 1:
            cpu = {"value": sub.n_reads / dt_cpu, "unit": UNIT, "cores": cores, "kind": "port", "simd": "avx2 int16",
                   "sample": f"first {sub.n_loci} loci ({sub.n_reads} reads) of batch 0, {dt_cpu:.2f} s, "
                             f"{cells / dt_cpu / 1e9:.2f} GCUPS reference-equivalent",
                   "gcups": cells / dt_cpu / 1e9}
        eng.run(dev_batches[0], params, kernel, stream)
        got = eng.download(dev_batches[0])[:sub.n_reads]
        parity = {"bit_exact": bool(np.array_equal(got, want)), "reads_compared": int(sub.n_reads)}
        if ref_sets:
            rb, start, ref_size, rc, anchor, _ = ref_sets[0]
            got_ref = eng.ref_counts(rb, start, ref_size, rc, anchor)
            arena = rb.arena.tobytes().decode()
            n_chk = min(512, rb.n_loci)
            ok = True
            for l in range(n_chk):
                o, (fl, tr, fr) = int(rb.seq_off[l]), (int(v) for v in rb.lens[l])
                mo, ml = int(rb.motif_off[l]), int(rb.motif_len[l])
                (cn, score), lo, ro, (n_off, n_fin), (fl2, _, fr2) = orc.get_ref_repeat_count(
                    int(start[l]), arena[o + fl:o + fl + tr], arena[o:o + fl], arena[o + fl + tr:o + fl + tr + fr],
                    arena[mo:mo + ml], int(ref_size[l]), anchor, 250, 3, 1)
                ok = ok and got_ref[l].tolist() == [cn, score, lo, ro, n_off, n_fin, len(fl2), len(fr2)]
            ref_parity = {"bit_exact": bool(ok), "loci_compared": n_chk}

    if rank == 0:
        steps = max(1, args.steps)
        dp_s = agg2["dp_ms"] * 1e-3
        # dominant kernel = the DP kernel of the read path; algorithmic work = 4 int32 ops per executed cell; kernel
        # time from the read-path-only region (in region 1 the kernels share the SMs with the reference windows)
        achieved = agg2["executed_cells"] * 4.0 / dp_s / 1e12 if dp_s > 0 else 0.0
        peaks_file = os.path.join(ROOT, "MEASURED_PEAKS.json")
        hbm_peak = json.load(open(peaks_file)).get("hbm_gbs") if os.path.exists(peaks_file) else 6650.0
        arena_gbs = (reads_per_step * 300.0 * args.steps) / dp_s / 1e9 if dp_s > 0 else 0.0
        traffic, traffic_src = ncu_dram_traffic()
        n_dp_reads = agg2["reads_packed_kernel"] + agg2["reads_general_kernel"]
        ref_dp_s = ref_solo["dp_ms"] * 1e-3
        cfg = config_dict(args, world)
        cfg["host_affinity"] = numa_note
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": elapsed_ms / steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int32" if args.kernel == "general" else "u16x2/int32",
            "data": "synthetic", "config": cfg,
            "value_is": "whole hot path of a block of loci: get_ref_repeat_count once per locus (host arrays, second native "
                        "context, running under the read kernels) + get_repeat_count per read (batch resident in HBM)"
                        if ref_sets else "read path only (--no-ref-path)",
            "reads_only": {"value": total_reads / (reads_only_ms * 1e-3), "unit": UNIT, "ms_per_step": reads_only_ms / steps},
            "sustained": sustained,
            "gcups_executed": exec_cells / (elapsed_ms * 1e-3) / 1e9,
            "gcups_reference_equivalent": ref_cells / (elapsed_ms * 1e-3) / 1e9,
            "roofline": {"bound": "int_alu", "achieved": achieved, "peak": peak["dual_pipe"], "unit": "Tiop/s",
                         "frac": achieved / peak["dual_pipe"] if peak["dual_pipe"] else None, "traffic": traffic,
                         "traffic_note": f"DRAM bytes ({traffic_src})" if traffic else None,
                         "kernel": "dp_general_kernel" if agg["reads_packed_kernel"] == 0 else "dp_packed_kernel",
                         "ops_per_cell": 4, "kernel_ms_per_step": agg2["dp_ms"] / steps,
                         "kernel_share_of_step": agg2["dp_ms"] / reads_only_ms if reads_only_ms else None,
                         "measured_in": "the read-path-only region (reads_only)",
                         "cells_are": "executed cells of the DISTINCT reads (identical reads of a locus share one table)",
                         "distinct_reads_per_step": n_dp_reads / steps,
                         "peak_how": "measured now on this GPU: lane-level 32-bit integer instructions/s, "
                                     "VIADDMNMX + IMAD chains on both issue pipes (ALU-pipe only: "
                                     f"{peak['alu_pipe']:.2f}, FMA-pipe only: {peak['fma_pipe']:.2f})",
                         "hbm": {"achieved": arena_gbs, "peak": hbm_peak, "unit": "GB/s",
                                 "note": "arena streaming only; the path is INT-ALU bound, not HBM bound"}},
            "ref_path": None if not ref_sets else {
                "ms_per_step": (elapsed_ms - reads_only_ms) / steps, "ms_per_step_is": "added to the read path's step by the "
                "reference windows running under it (alone: tools/bench_ref_path.py)", "loci_per_step": args.loci_per_step,
                "share_of_hot_path_time": (elapsed_ms - reads_only_ms) / elapsed_ms,
                "share_of_executed_cells": agg_ref["executed_cells"] / max(1.0, agg["executed_cells"] + agg_ref["executed_cells"]),
                "alone_ms_per_block": ref_solo_ms, "dp_kernel_ms_per_block_alone": ref_solo["dp_ms"],
                "replay_ms_per_block_alone": ref_solo["replay_ms"],
                "kernel_launches_per_step": agg_ref["kernel_launches"] / steps,
                "roofline": {"bound": "int_alu", "unit": "Tiop/s", "peak": peak["dual_pipe"], "measured": "alone, 4 blocks",
                             "achieved": ref_solo["executed_cells"] * 4.0 / ref_dp_s / 1e12 if ref_dp_s > 0 else None,
                             "frac": ref_solo["executed_cells"] * 4.0 / ref_dp_s / 1e12 / peak["dual_pipe"] if ref_dp_s > 0 else None,
                             "kernel": "dp_packed_kernel (reference mode: both sg_qe sweeps of a locus) + the final count"},
                "parity_sample": ref_parity,
                "how": "Engine.ref_counts: host arrays in / 8 ints per locus out, one call per block"},
            "cpu_baseline": cpu, "e2e": e2e,
            "gpu_launches": int(agg["kernel_launches"] + agg_ref["kernel_launches"]),
            "replay_ms_per_step": agg["replay_ms"] / steps,
            "widening_passes": int(agg["widening_passes"]),
            "reads_packed_kernel": int(agg["reads_packed_kernel"]),
            "reads_general_kernel": int(agg["reads_general_kernel"]),
            # rank 0's share, like the two counters above (identical reads of a locus run the DP once)
            "reads_deduped": max(0, int(reads_per_step * args.steps - n_dp_reads)),
            "parity_sample_bit_exact": parity["bit_exact"] if parity else None, "parity_sample": parity, "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
