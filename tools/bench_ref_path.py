#!/usr/bin/env python
"""Throughput of the reference-genome path (get_ref_repeat_count, strkit/call/repeats.py:73-192, once per locus)
next to the read path it precedes in call_locus: loci/s of strk_ref_counts on a block of synthetic loci whose
reference window is an error-free copy of the locus (one sequence per locus), checked against the CPU oracle.

    python tools/bench_ref_path.py [n_loci] [--mixed-tiers] [--reps N]

--mixed-tiers: the rows of search parameters cycle over the four tiers of repeat_count_params.py:17-42 (a block
whose loci span them, as BlockSession sends it) instead of all using the first one.  The call is timed N times
(default 10) after a warm-up; the median is reported.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

# (max_iters, local search range, step size) below 200, from 200, 1000 and 2000 reference copies
TIERS = np.array([[250, 3, 1], [200, 3, 3], [150, 3, 5], [50, 1, 15]], dtype=np.int32)


def main():
    import torch

    import strkit_b200
    from strkit_b200 import synth
    from strkit_b200.batcher import ReadBatch
    from tests import oracle_lib

    ap = argparse.ArgumentParser()
    ap.add_argument("n_loci", nargs="?", type=int, default=32768)
    ap.add_argument("--mixed-tiers", action="store_true")
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    n_loci = args.n_loci
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    rb = synth.generate(synth.CONFIGS[2], n_loci, seed=77, device=dev).to_host()
    first = rb.read_begin[:-1]  # the first read of every locus plays the reference window
    # compact arena of its own: [reference windows][motifs]
    lens = rb.lens[first].copy()
    tot = lens.sum(axis=1).astype(np.int64)
    seq_off = np.concatenate([[0], np.cumsum(tot)[:-1]]).astype(np.uint64)
    src = np.repeat(rb.seq_off[first].astype(np.int64) - seq_off.astype(np.int64), tot) + np.arange(int(tot.sum()))
    ml = rb.motif_len.astype(np.int64)
    motif_off = (int(tot.sum()) + np.concatenate([[0], np.cumsum(ml)[:-1]])).astype(np.uint64)
    msrc = np.repeat(rb.motif_off.astype(np.int64) - (motif_off.astype(np.int64)), ml) + int(tot.sum()) + np.arange(int(ml.sum()))
    arena = np.concatenate([rb.arena[src], rb.arena[msrc]])
    ref = ReadBatch(arena=arena, seq_off=seq_off, lens=lens, est_cn=rb.est_cn[first].copy(),
                    read_begin=np.arange(n_loci + 1, dtype=np.int64), motif_off=motif_off, motif_len=rb.motif_len)
    start = ref.est_cn.copy()
    ref_size = ref.lens[:, 1].copy()
    rc = TIERS[np.arange(n_loci) % len(TIERS)] if args.mixed_tiers else np.tile(TIERS[0], (n_loci, 1))
    rc = np.ascontiguousarray(rc)
    eng = strkit_b200.Engine()
    eng.ref_counts(ref, start, ref_size, rc, 5)  # grows the recycled device buffers to block size
    times = []
    for _ in range(max(1, args.reps)):
        t0 = time.perf_counter()
        out = eng.ref_counts(ref, start, ref_size, rc, 5)
        times.append(time.perf_counter() - t0)
    dt = float(np.median(times))
    st = eng.stats()
    params = strkit_b200.RepeatCountParams("repalign", 50, 3, 1)
    rbp = synth.generate(synth.CONFIGS[2], n_loci, seed=77, device=dev).to_host(pin=True)
    eng.count_reads(rbp, params)
    t1 = time.perf_counter()
    eng.count_reads(rbp, params)
    dt_reads = time.perf_counter() - t1
    orc = oracle_lib.load()
    ok = True
    tc = time.perf_counter()
    n_chk = 128
    arena = ref.arena.tobytes()
    for l in range(n_chk):
        o, (fl, tr, fr) = int(ref.seq_off[l]), ref.lens[l]
        s = arena[o:o + fl + tr + fr].decode()
        mo, ml = int(ref.motif_off[l]), int(ref.motif_len[l])
        (cn, score), lo, ro, (n_off, n_fin), (fl2, tr2, fr2) = orc.get_ref_repeat_count(
            int(start[l]), s[fl:fl + tr], s[:fl], s[fl + tr:], arena[mo:mo + ml].decode(), int(ref_size[l]), 5, *rc[l].tolist())
        ok = ok and out[l].tolist() == [cn, score, lo, ro, n_off, n_fin, len(fl2), len(fr2)]
    dt_cpu = time.perf_counter() - tc
    print(json.dumps({"n_loci": n_loci, "tiers": 4 if args.mixed_tiers else 1, "ref_path_s": dt,
                      "ref_ms_per_call": [round(t * 1e3, 3) for t in times], "ref_loci_per_s": n_loci / dt,
                      "widening_passes": int(st["widening_passes"]),
                      "read_path_same_loci_s": dt_reads, "ref_share_of_locus_block": dt / (dt + dt_reads),
                      "parity_sample_bit_exact": bool(ok), "cpu_oracle_loci_per_s_1core": n_chk / dt_cpu}))


if __name__ == "__main__":
    main()
