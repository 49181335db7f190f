#!/usr/bin/env python
"""Allele calls for deep loci: strk_call_alleles_ploidy on loci of 256, 257, 1000, 5000 and 20 000 reads, A = 2 and 4.

    python tools/bench_alleles_deep.py > profiles/r3_alleles_deep.json

256 reads is the largest shallow locus (one thread per replicate), 257 the smallest deep one (one warp per
replicate), so that pair shows what the switch costs.  Workload per row: about --reads reads in loci of one depth
(at least 8 loci), A distinct alleles drawn from 8..80 at least 3 copies apart, +-1 stutter on 6 % of reads, uniform
weights; 1000 replicates, n_init 3.  Reported per row: kernel ms (CUDA events around the kernels), wall ms of the
call, loci/s on the kernel time; the checker (numpy + scikit-learn, oracle/alleles_oracle.py) on a sample of loci,
one process per core, at --cpu-bootstrap replicates (stated in the row).  The GPU's name and power limit are read
in the same run.
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def make_loci(rng, n_loci, depth, A):
    rb = np.arange(n_loci + 1, dtype=np.int64) * depth
    alleles = 8 + 3 * np.sort(np.stack([rng.choice(25, size=A, replace=False) for _ in range(n_loci)]), axis=1)
    locus = np.repeat(np.arange(n_loci), depth)
    cn = alleles[locus, rng.integers(0, A, size=locus.shape[0])] + rng.choice([-1, 0, 1], size=locus.shape[0],
                                                                               p=[.03, .94, .03])
    return cn.astype(np.int32), np.full(locus.shape[0], 1.0 / depth), rb


def _checker_one(job):
    from oracle import alleles_oracle as ao

    cn, A, num_bootstrap, seed = job
    ao.call_alleles(cn, np.full(len(cn), 1.0 / len(cn)), A, 4, seed, ao.OracleParams(num_bootstrap=num_bootstrap))


def gpu_context():
    import torch

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--depths", default="256,257,1000,5000,20000")
    ap.add_argument("--alleles", default="2,4")
    ap.add_argument("--reads", type=int, default=500_000, help="reads per row (loci = reads / depth, at least 8)")
    ap.add_argument("--bootstrap", type=int, default=1000)
    ap.add_argument("--n-init", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cpu-bootstrap", type=int, default=100)
    ap.add_argument("--cpu-sample-loci", type=int, default=0, help="per row; default: one per host core")
    args = ap.parse_args()

    import strkit_b200
    from strkit_b200 import alleles

    eng = strkit_b200.Engine()
    cores = os.cpu_count() or 1
    sample = args.cpu_sample_loci or cores
    kw = dict(num_bootstrap=args.bootstrap, n_init=args.n_init, seed=1234, engine=eng)
    out = {**gpu_context(), "num_bootstrap": args.bootstrap, "n_init": args.n_init, "reads_per_row": args.reads,
           "checker_cores": cores, "checker_num_bootstrap": args.cpu_bootstrap, "rows": []}
    for A in [int(a) for a in args.alleles.split(",")]:
        for depth in [int(d) for d in args.depths.split(",")]:
            n_loci = max(8, args.reads // depth)
            rng = np.random.default_rng(9000 + 10 * A + depth)
            cn, w, rb = make_loci(rng, n_loci, depth, A)
            alleles.call_alleles_ploidy_batch(cn[:rb[2]], w[:rb[2]], rb[:3], A, **kw)  # warm-up, buffers
            best = None
            for _ in range(args.reps):
                t0 = time.perf_counter()
                r = alleles.call_alleles_ploidy_batch(cn, w, rb, A, **kw)
                wall = (time.perf_counter() - t0) * 1e3
                if best is None or r.kernel_ms < best[0].kernel_ms:
                    best = (r, wall)
            r, wall = best
            row = {"A": A, "reads_per_locus": depth, "loci": n_loci, "path": "deep" if depth > 256 else "shallow",
                   "kernel_ms": r.kernel_ms, "wall_ms": wall, "loci_per_s_kernel": n_loci / (r.kernel_ms / 1e3),
                   "status_counts": {str(k): int(v) for k, v in zip(*np.unique(r.status, return_counts=True))},
                   "modal_n_counts": {str(k): int(v) for k, v in zip(*np.unique(r.modal_n, return_counts=True))}}
            ns = min(sample, n_loci)
            jobs = [(cn[rb[l]:rb[l + 1]].copy(), A, args.cpu_bootstrap, 1234 + l) for l in range(ns)]
            t0 = time.perf_counter()
            with mp.get_context("fork").Pool(cores) as pool:
                pool.map(_checker_one, jobs)
            t_cpu = time.perf_counter() - t0
            row["checker"] = {"sample_loci": ns, "num_bootstrap": args.cpu_bootstrap, "s": t_cpu,
                              "loci_per_s": ns / t_cpu}
            out["rows"].append(row)
            print(json.dumps(row), file=sys.stderr, flush=True)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
