#!/usr/bin/env python
"""Allele calls per allele count: strk_call_alleles_ploidy on loci of A true alleles, A = 1, 2, 3, 4, 6, 8.

    python tools/bench_alleles_ploidy.py > alleles_ploidy.json

Workload: --loci loci of about 30 reads (24..36) per A, alleles drawn from 8..60 (repeats allowed, i.e. dosage),
+-1 stutter on 6 % of reads, uniform read weights; the config-5 settings (1000 replicates, n_init 3).  Reported:
  * per A: kernel ms (CUDA events around the kernels), wall ms of the call, loci/s on the kernel time;
  * at A = 2: the uniform entry (strk_call_alleles) and the per-locus one on the same batch and seed, whether their
    outputs are byte-identical, and both times;
  * the checker (numpy + scikit-learn, oracle/alleles_oracle.py) on a sample of loci per A, one process per core.
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def make_loci(rng, n_loci, A):
    n = rng.integers(24, 37, size=n_loci)
    rb = np.concatenate([[0], np.cumsum(n)]).astype(np.int64)
    alleles = np.sort(rng.integers(8, 61, size=(n_loci, A)), axis=1)
    locus = np.repeat(np.arange(n_loci), n)
    cn = alleles[locus, rng.integers(0, A, size=locus.shape[0])] + rng.choice([-1, 0, 1], size=locus.shape[0],
                                                                               p=[.03, .94, .03])
    w = 1.0 / np.repeat(n, n).astype(np.float64)
    return cn.astype(np.int32), w, rb


def _checker_one(job):
    from oracle import alleles_oracle as ao

    cn, A, num_bootstrap, seed = job
    ao.call_alleles(cn, np.full(len(cn), 1.0 / len(cn)), A, 4, seed, ao.OracleParams(num_bootstrap=num_bootstrap))


def timed(fn, reps):
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        r = fn()
        wall = (time.perf_counter() - t0) * 1e3
        if best is None or r.kernel_ms < best[0].kernel_ms:
            best = (r, wall)
    return best


def same_rows(x, y, a):
    return all(np.asarray(getattr(x, f))[..., :a].tobytes() == np.asarray(getattr(y, f))[..., :a].tobytes()
               for f in ("call", "call_95_cis", "call_99_cis", "means", "weights", "stdevs")) and \
        x.modal_n.tobytes() == y.modal_n.tobytes() and x.status.tobytes() == y.status.tobytes()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--loci", type=int, default=100_000)
    ap.add_argument("--alleles", default="1,2,3,4,6,8")
    ap.add_argument("--bootstrap", type=int, default=1000)
    ap.add_argument("--n-init", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cpu-sample-loci", type=int, default=0, help="per A; default: one per host core")
    args = ap.parse_args()
    import torch

    import strkit_b200
    from strkit_b200 import alleles

    eng = strkit_b200.Engine()
    cores = os.cpu_count() or 1
    sample = args.cpu_sample_loci or cores
    kw = dict(num_bootstrap=args.bootstrap, n_init=args.n_init, seed=1234, engine=eng)
    out = {"gpu": torch.cuda.get_device_name(0), "loci": args.loci, "num_bootstrap": args.bootstrap,
           "n_init": args.n_init, "reads_per_locus": "24..36", "per_A": [], "checker_cores": cores}
    for A in [int(a) for a in args.alleles.split(",")]:
        rng = np.random.default_rng(7000 + A)
        cn, w, rb = make_loci(rng, args.loci, A)
        alleles.call_alleles_ploidy_batch(cn[:rb[64]], w[:rb[64]], rb[:65], A, **kw)  # warm-up, buffers
        r, wall = timed(lambda: alleles.call_alleles_ploidy_batch(cn, w, rb, A, **kw), args.reps)
        row = {"A": A, "kernel_ms": r.kernel_ms, "wall_ms": wall, "loci_per_s_kernel": args.loci / (r.kernel_ms / 1e3),
               "status_counts": {str(k): int(v) for k, v in zip(*np.unique(r.status, return_counts=True))},
               "modal_n_counts": {str(k): int(v) for k, v in zip(*np.unique(r.modal_n, return_counts=True))}}
        if A == 2:
            old, wall_old = timed(lambda: alleles.call_alleles_batch(cn, w, rb, 2, **kw), args.reps)
            row["uniform_entry"] = {"kernel_ms": old.kernel_ms, "wall_ms": wall_old,
                                    "outputs_byte_identical": same_rows(old, r, 2)}
        jobs = [(cn[rb[l]:rb[l + 1]].copy(), A, args.bootstrap, 1234 + l) for l in range(sample)]
        t0 = time.perf_counter()
        with mp.get_context("fork").Pool(cores) as pool:
            pool.map(_checker_one, jobs)
        t_cpu = time.perf_counter() - t0
        row["checker"] = {"sample_loci": sample, "s": t_cpu, "loci_per_s": sample / t_cpu}
        out["per_A"].append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
