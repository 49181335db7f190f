"""Bootstrap + Gaussian-mixture allele calls on the GPU: the consumer of the per-read repeat counts.

Mirrors the reference's `call_alleles` (strkit/call/allele.py:176-336) and, batched over many loci,
the loop `call_locus` runs around it (call_alleles_with_gmm, call_locus.py:177-219).  The arithmetic is in
the native library (csrc/alleles.cuh): one CUDA thread per (locus, bootstrap replicate) resamples, seeds
with k-means++, runs sklearn's EM in float64 and applies the reference's peak filters (one warp per replicate
for loci of more than 256 reads); one CTA per locus sorts the replicate estimates and takes medians /
confidence intervals.

The random streams are the library's own (counter-based, keyed by seed / locus / replicate), so calls and
intervals agree with the reference statistically (tests/test_alleles_*.py state the tolerance), while
everything that is deterministic given the random choices is checked exactly.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Sequence

import numpy as np

from ._native import check, lib
from .engine import Engine, default_engine

__all__ = ["AlleleCalls", "CallData", "call_alleles_batch", "call_alleles_ploidy_batch", "call_alleles", "gmm_fit_counts",
           "gmm_fit_counts_ploidy", "gmm_fit_counts_deep", "aggregate_replicates"]


def _p(a: np.ndarray) -> int:
    return a.ctypes.data


@dataclass
class AlleleCalls:
    """Per-locus results of a batch; row l is meaningful where status[l] is 0 or 2 (1 = fewer than min_reads reads, the
    reference returns None; 2 = single distinct copy number, no bootstrap; 3 = fewer reads than alleles, where the
    reference raises).  With per-locus allele counts the arrays are n_alleles.max() wide and locus l uses the
    first n_alleles[l] columns (the rest are 0)."""
    call: np.ndarray          # int32  [n_loci, n_alleles]
    call_95_cis: np.ndarray   # int32  [n_loci, n_alleles, 2]
    call_99_cis: np.ndarray   # int32  [n_loci, n_alleles, 2]
    means: np.ndarray         # float64 [n_loci, n_alleles]
    weights: np.ndarray       # float64 [n_loci, n_alleles]
    stdevs: np.ndarray        # float64 [n_loci, n_alleles]
    modal_n: np.ndarray       # int32  [n_loci]
    status: np.ndarray        # int32  [n_loci]
    kernel_ms: float = 0.0
    n_alleles: np.ndarray | None = None  # int32 [n_loci]: per-locus allele counts (call_alleles_ploidy_batch)


@dataclass
class CallData:
    """Plain-Python stand-in for strkit_rust_ext.CallData as `call_alleles` constructs it
    (allele.py:207-215,324-336): same constructor keywords, same attribute names downstream code reads."""
    call: np.ndarray
    call_95_cis: np.ndarray
    call_99_cis: np.ndarray
    means: np.ndarray
    weights: np.ndarray
    stdevs: np.ndarray
    modal_n: int
    extra: dict = field(default_factory=dict)

    @property
    def peak_means(self):
        return self.means

    @property
    def peak_weights(self):
        return self.weights

    @property
    def peak_stdevs(self):
        return self.stdevs

    @property
    def peak_modal_n(self):
        return self.modal_n


def _unpack(out_i: np.ndarray, out_d: np.ndarray, status: np.ndarray, n_alleles: int, ms: float) -> AlleleCalls:
    a = n_alleles
    return AlleleCalls(call=out_i[:, 1:1 + a].copy(), call_95_cis=out_i[:, 1 + a:1 + 3 * a].reshape(-1, a, 2).copy(),
                       call_99_cis=out_i[:, 1 + 3 * a:1 + 5 * a].reshape(-1, a, 2).copy(), means=out_d[:, :a].copy(),
                       weights=out_d[:, a:2 * a].copy(), stdevs=out_d[:, 2 * a:3 * a].copy(), modal_n=out_i[:, 0].copy(),
                       status=status, kernel_ms=ms)


def call_alleles_batch(cn: np.ndarray, weights: np.ndarray, read_begin: np.ndarray, n_alleles: int = 2, *,
                       num_bootstrap: int = 100, min_reads: int = 4, min_allele_reads: int = 2,
                       force_gm_filter: bool = False, expansion_ratio: float = 5.0, filter_factor: int = 3,
                       n_init: int = 3, seed: int = 0, engine: Engine | None = None) -> AlleleCalls:
    """call_alleles for every locus of a batch.  cn / weights are per read (weights normalised per locus, as
    call_alleles_with_gmm does at call_locus.py:191-192), read_begin delimits the loci.  Defaults are the
    reference's (params.py:39-56,166-172)."""
    eng = engine or default_engine()
    cn = np.ascontiguousarray(cn, dtype=np.int32)
    weights = np.ascontiguousarray(weights, dtype=np.float64)
    read_begin = np.ascontiguousarray(read_begin, dtype=np.int64)
    n_loci = int(read_begin.shape[0]) - 1
    if n_loci < 0 or cn.shape != weights.shape or cn.ndim != 1:
        raise ValueError("call_alleles_batch: cn and weights must be flat arrays of equal length; read_begin [n_loci + 1]")
    out_i = np.zeros((max(n_loci, 0), 1 + 5 * n_alleles), dtype=np.int32)
    out_d = np.zeros((max(n_loci, 0), 3 * n_alleles), dtype=np.float64)
    status = np.zeros(max(n_loci, 0), dtype=np.int32)
    ms = np.zeros(1, dtype=np.float64)
    check(lib.strk_call_alleles(eng._ctx, _p(cn), _p(weights), _p(read_begin), n_loci, n_alleles, num_bootstrap,
                                min_reads, min_allele_reads, int(force_gm_filter), float(expansion_ratio), filter_factor,
                                n_init, int(seed) & 0xFFFFFFFFFFFFFFFF, _p(out_i), _p(out_d), _p(status), _p(ms)))
    return _unpack(out_i, out_d, status, n_alleles, float(ms[0]))


def call_alleles_ploidy_batch(cn: np.ndarray, weights: np.ndarray, read_begin: np.ndarray, n_alleles, *,
                              num_bootstrap: int = 100, min_reads: int = 4, min_allele_reads: int = 2,
                              force_gm_filter: bool = False, expansion_ratio: float = 5.0, filter_factor: int = 3,
                              n_init: int = 3, seed: int = 0, engine: Engine | None = None) -> AlleleCalls:
    """call_alleles_batch with an allele count per locus (1..8; an int applies to every locus), e.g. the
    `n_alleles` of each STRkitLocus as the ploidy config sets it.  One call serves a catalog of any mix of counts;
    loci with one or two alleles get the rows call_alleles_batch would give them (same seed, one chunk)."""
    eng = engine or default_engine()
    cn = np.ascontiguousarray(cn, dtype=np.int32)
    weights = np.ascontiguousarray(weights, dtype=np.float64)
    read_begin = np.ascontiguousarray(read_begin, dtype=np.int64)
    n_loci = int(read_begin.shape[0]) - 1
    if n_loci < 0 or cn.shape != weights.shape or cn.ndim != 1:
        raise ValueError("call_alleles_ploidy_batch: cn and weights must be flat arrays of equal length; "
                         "read_begin [n_loci + 1]")
    a_loc = np.ascontiguousarray(np.broadcast_to(np.asarray(n_alleles, dtype=np.int32), (n_loci,)))
    s = max(1, int(a_loc.max(initial=1)))
    out_i = np.zeros((n_loci, 1 + 5 * s), dtype=np.int32)
    out_d = np.zeros((n_loci, 3 * s), dtype=np.float64)
    status = np.zeros(n_loci, dtype=np.int32)
    ms = np.zeros(1, dtype=np.float64)
    check(lib.strk_call_alleles_ploidy(eng._ctx, _p(cn), _p(weights), _p(read_begin), n_loci, _p(a_loc), num_bootstrap,
                                       min_reads, min_allele_reads, int(force_gm_filter), float(expansion_ratio),
                                       filter_factor, n_init, int(seed) & 0xFFFFFFFFFFFFFFFF, _p(out_i), _p(out_d),
                                       _p(status), _p(ms)))
    res = _unpack(out_i, out_d, status, s, float(ms[0]))
    res.n_alleles = a_loc
    return res


def call_alleles(repeats_fwd, repeats_rev, read_weights_fwd, read_weights_rev, params, min_reads: int, n_alleles: int,
                 separate_strands: bool, read_bias_corr_min: int, seed: int | None, logger_=None, debug_str: str = "",
                 engine: Engine | None = None) -> CallData | None:
    """Drop-in for strkit.call.allele.call_alleles (allele.py:176-189): same arguments, same return shape.
    `params` needs num_bootstrap, min_allele_reads, force_gm_filter and gmm_params (n_init, expansion_ratio,
    filter_factor), i.e. a reference CallParams works unchanged."""
    if separate_strands:
        # both reference call sites pass False (call_locus.py:209,263); the strand-balanced branch is not built
        raise NotImplementedError("call_alleles: separate_strands=True is not implemented on the GPU path")
    cn = np.concatenate((np.asarray(repeats_fwd, dtype=np.int32).ravel(), np.asarray(repeats_rev, dtype=np.int32).ravel()))
    w = np.concatenate((np.asarray(read_weights_fwd, dtype=np.float64).ravel(),
                        np.asarray(read_weights_rev, dtype=np.float64).ravel()))
    gp = params.gmm_params
    batch = call_alleles_batch if n_alleles <= 2 else call_alleles_ploidy_batch
    res = batch(cn, w, np.array([0, cn.shape[0]], dtype=np.int64), n_alleles, num_bootstrap=params.num_bootstrap,
                min_reads=min_reads, min_allele_reads=params.min_allele_reads, force_gm_filter=params.force_gm_filter,
                expansion_ratio=gp.expansion_ratio, filter_factor=gp.filter_factor, n_init=gp.n_init,
                seed=0 if seed is None else int(seed), engine=engine)
    if res.status[0] == 1:
        return None
    if res.status[0] == 3:  # scikit-learn's GaussianMixture.fit raises this inside the reference's call_alleles
        raise ValueError(f"Expected n_samples >= n_components but got n_components = {n_alleles}, "
                         f"n_samples = {cn.shape[0]}")
    return CallData(call=res.call[0], call_95_cis=res.call_95_cis[0], call_99_cis=res.call_99_cis[0], means=res.means[0],
                    weights=res.weights[0], stdevs=res.stdevs[0], modal_n=int(res.modal_n[0]))


def gmm_fit_counts(values: Sequence[np.ndarray], counts: Sequence[np.ndarray], init: np.ndarray, n_alleles: int = 2, *,
                   num_bootstrap: int = 100, min_allele_reads: int = 2, force_gm_filter: bool = False,
                   expansion_ratio: float = 5.0, filter_factor: int = 3, engine: Engine | None = None) -> np.ndarray:
    """fit_gmm + per-replicate bookkeeping (allele.py:56-123,249-293) for explicit replicates and explicit
    k-means++ seeds: problem q has distinct values values[q] (ascending) with multiplicities counts[q];
    init[q, t] = (i0, i1) indices into values[q] for restart t.  Returns [q, 7] =
    (mean0, weight0, stdev0, mean1, weight1, stdev1, n_peaks)."""
    eng = engine or default_engine()
    nq = len(values)
    init = np.ascontiguousarray(init, dtype=np.int32).reshape(nq, -1, 2)
    n_init = init.shape[1]
    kcap = max(1, max((len(v) for v in values), default=1))
    x = np.zeros((nq, kcap), dtype=np.float64)
    c = np.zeros((nq, kcap), dtype=np.int32)
    k = np.zeros(nq, dtype=np.int32)
    for q, (v, cc) in enumerate(zip(values, counts)):
        k[q] = len(v)
        x[q, :len(v)] = v
        c[q, :len(v)] = cc
    out = np.zeros((nq, 7), dtype=np.float64)
    check(lib.strk_gmm_fit_counts(eng._ctx, _p(x), _p(c), _p(k), _p(init), nq, kcap, n_alleles, num_bootstrap,
                                  min_allele_reads, int(force_gm_filter), float(expansion_ratio), filter_factor, n_init,
                                  _p(out)))
    return out


def gmm_fit_counts_ploidy(values: Sequence[np.ndarray], counts: Sequence[np.ndarray], n_alleles,
                          init: Sequence[np.ndarray] | None = None, *, n_init: int = 3, num_bootstrap: int = 100,
                          min_allele_reads: int = 2, force_gm_filter: bool = False, expansion_ratio: float = 5.0,
                          filter_factor: int = 3, seed: int = 0, engine: Engine | None = None) -> np.ndarray:
    """gmm_fit_counts for problems with their own allele counts (n_alleles: an int or one per problem, 1..8).
    init[q] (None: k-means++ draws) holds the forced seeds of every fit fit_gmm's staged loop may run on problem q:
    for nc = A, A-1, ..., 2, n_init rows of nc indices into values[q], flattened.  Returns [q, 3 * S + 1] with
    S = max(n_alleles): means[S], weights[S], stdevs[S] (the first A[q] sorted by mean, the rest 0), n_peaks.
    Entries beyond the fitted n_peaks are random copies of fitted components (the reference's fill)."""
    return _fit_counts(lib.strk_gmm_fit_counts_ploidy, values, counts, n_alleles, init, n_init, num_bootstrap,
                       min_allele_reads, force_gm_filter, expansion_ratio, filter_factor, seed, engine)


def gmm_fit_counts_deep(values: Sequence[np.ndarray], counts: Sequence[np.ndarray], n_alleles,
                        init: Sequence[np.ndarray] | None = None, *, n_init: int = 3, num_bootstrap: int = 100,
                        min_allele_reads: int = 2, force_gm_filter: bool = False, expansion_ratio: float = 5.0,
                        filter_factor: int = 3, seed: int = 0, engine: Engine | None = None) -> np.ndarray:
    """gmm_fit_counts_ploidy through the warp-cooperative fit that deep loci (more than 256 reads) use: the same
    arguments and output, for up to 4096 distinct values per problem and any number of points.  Without forced
    seeds its k-means++ draws come from another stream than gmm_fit_counts_ploidy's."""
    return _fit_counts(lib.strk_gmm_fit_counts_deep, values, counts, n_alleles, init, n_init, num_bootstrap,
                       min_allele_reads, force_gm_filter, expansion_ratio, filter_factor, seed, engine)


def _fit_counts(fn, values, counts, n_alleles, init, n_init, num_bootstrap, min_allele_reads, force_gm_filter,
                expansion_ratio, filter_factor, seed, engine):
    name = fn.__name__[len("strk_"):]
    eng = engine or default_engine()
    nq = len(values)
    a = np.ascontiguousarray(np.broadcast_to(np.asarray(n_alleles, dtype=np.int32), (nq,)))
    s = max(1, int(a.max(initial=1)))
    kcap = max(1, max((len(v) for v in values), default=1))
    x = np.zeros((nq, kcap), dtype=np.float64)
    c = np.zeros((nq, kcap), dtype=np.int32)
    k = np.zeros(nq, dtype=np.int32)
    for q, (v, cc) in enumerate(zip(values, counts)):
        k[q] = len(v)
        x[q, :len(v)] = v
        c[q, :len(v)] = cc
    if init is not None:
        init = [np.asarray(i, dtype=np.int32).ravel() for i in init]
        for q, i in enumerate(init):
            want = n_init * (int(a[q]) * (int(a[q]) + 1) // 2 - 1) if 1 <= a[q] <= 8 else i.size
            if i.size != want:
                raise ValueError(f"{name}: problem {q} has {i.size} seed indices, expected {want}")
        init = np.ascontiguousarray(np.concatenate(init) if init else np.zeros(0, dtype=np.int32), dtype=np.int32)
    out = np.zeros((nq, 3 * s + 1), dtype=np.float64)
    check(fn(eng._ctx, _p(x), _p(c), _p(k), _p(a), None if init is None else _p(init), nq, kcap, num_bootstrap,
             min_allele_reads, int(force_gm_filter), float(expansion_ratio), filter_factor, n_init,
             int(seed) & 0xFFFFFFFFFFFFFFFF, _p(out)))
    return out


def aggregate_replicates(rep_means: np.ndarray, rep_weights: np.ndarray, rep_stdevs: np.ndarray, rep_peaks: np.ndarray,
                         engine: Engine | None = None) -> AlleleCalls:
    """The aggregation of call_alleles (allele.py:295-336) for replicate arrays [n_loci, n_alleles, num_bootstrap]
    (rep_peaks [n_loci, num_bootstrap])."""
    eng = engine or default_engine()
    rm = np.ascontiguousarray(rep_means, dtype=np.float64)
    rw = np.ascontiguousarray(rep_weights, dtype=np.float64)
    rs = np.ascontiguousarray(rep_stdevs, dtype=np.float64)
    rp = np.ascontiguousarray(rep_peaks, dtype=np.uint8)
    n_loci, a, b = rm.shape
    out_i = np.zeros((n_loci, 1 + 5 * a), dtype=np.int32)
    out_d = np.zeros((n_loci, 3 * a), dtype=np.float64)
    check(lib.strk_alleles_aggregate(eng._ctx, _p(rm), _p(rw), _p(rs), _p(rp), n_loci, a, b, _p(out_i), _p(out_d)))
    return _unpack(out_i, out_d, np.zeros(n_loci, dtype=np.int32), a, 0.0)
