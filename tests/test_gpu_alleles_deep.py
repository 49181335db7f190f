"""GPU tests of allele calls for deep loci (more than 256 reads): the warp-cooperative fit (strk_gmm_fit_counts_deep)
and its routing inside strk_call_alleles / strk_call_alleles_ploidy, against the checker (oracle/alleles_oracle.py =
numpy + scikit-learn 1.9.0) and against the shallow path's own rows.

What is exact and what is statistical:
  * the warp fit given forced seeds: scikit-learn run stage by stage from the same seeds, to 1e-6 (or _tie_tol);
  * shallow rows of a batch with deep loci: byte-identical to the same batch without them;
  * deep rows: byte-identical from call to call with the same seed;
  * deep calls draw their own random numbers, so they are compared with the checker statistically.
"""
import dataclasses

import numpy as np
import pytest

from oracle import alleles_oracle as ao
from tests.test_gpu_alleles_ploidy import (_expected_outcomes, _fields, _matches_fitted_part, _poly_loci,
                                           _poly_replicate)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def al():
    import strkit_b200
    from strkit_b200 import alleles

    assert strkit_b200.device_count() > 0, "no CUDA device: these tests need a B200"
    return alleles


def _wide_replicate(rng, K, n):
    """K distinct values (a few clusters spread over a wide range) and n >= K points, every value present."""
    centres = np.sort(rng.choice(np.arange(20, 20 + 4 * K), size=int(rng.integers(2, 6)), replace=False))
    pool = np.unique(np.concatenate([c + np.arange(-K, K) for c in centres]))
    pool = pool[pool > 0]
    near = np.argsort(np.min(np.abs(pool[:, None] - centres[None, :]), axis=1), kind="stable")[:K]
    v = np.sort(pool[near])
    c = np.ones(K, dtype=np.int64)
    d = np.min(np.abs(v[:, None] - centres[None, :]), axis=1)
    p = np.exp(-d / max(2.0, K / 40))
    c += rng.multinomial(n - K, p / p.sum())
    return v, c


def test_deep_fits_match_sklearn_given_the_seeds(al):
    """Replicates with K in {2, 5, 40, 257, 1000, 4096} distinct values and 10 to 50 000 points, A in {2, 3, 4, 8}.
    Every fit of every stage is scikit-learn from the same forced seeds; the GPU row must match one acceptable branch,
    and over all A the four outcomes of fit_gmm's staged loop must occur."""
    rng = np.random.default_rng(2048)
    n_init = 3
    outcomes = set()
    for A in (2, 3, 4, 8):
        for nb, small in ((100, 60), (3, 30)):
            p = ao.OracleParams(num_bootstrap=nb)
            allele_filter = (p.min_allele_reads - 0.1) / nb
            values, counts, inits, accept = [], [], [], []
            reps = [_poly_replicate(rng, A) for _ in range(small)]
            if nb == 100:
                for K, n in ((2, 10), (5, 40), (40, 1000), (257, 3000), (1000, 20000), (4096, 50000)):
                    v, c = _wide_replicate(rng, K, n) if K > 5 else (np.arange(30, 30 + 3 * K, 3),
                                                                     1 + rng.multinomial(n - K, np.full(K, 1 / K)))
                    reps.append(np.repeat(v, c).astype(np.int32))
            for rep in reps:
                v, c = np.unique(rep, return_counts=True)
                seeds = {nc: [rng.choice(len(v), size=nc, replace=len(v) < nc) for _ in range(n_init)]
                         for nc in range(A, 1, -1)}
                accept.append(_expected_outcomes(rep, v, c, A, seeds, p, allele_filter))
                values.append(v.astype(np.float64)), counts.append(c.astype(np.int32))
                inits.append(np.concatenate([np.concatenate(seeds[nc]) for nc in range(A, 1, -1)]))
            got = al.gmm_fit_counts_deep(values, counts, A, inits, n_init=n_init, num_bootstrap=nb, seed=A)
            assert got.shape == (len(reps), 3 * A + 1)
            for q in range(len(reps)):
                ok = [w for w in accept[q] if _matches_fitted_part(got[q], A, A, w)]
                assert ok, (A, nb, q, len(values[q]), int(counts[q].sum()), got[q], accept[q])
                outcomes.add(ok[0][4])
    assert outcomes == {"kept", "dropped", "single", "last_fit"}, outcomes


@pytest.mark.parametrize("scale", [1, 1000])
def test_duplicate_centres_from_warp_kmeanspp(al, scale):
    """GaussianMixture(4) on [10] * 3 + [12] * 2 + [30] (each count times `scale`): the fourth k-means++ centre lands
    on point 0 and two components on 10 stay equal.  The warp's own k-means++ must give scikit-learn's result."""
    from sklearn.mixture import GaussianMixture

    rep = np.repeat([10.0, 12.0, 30.0], np.array([3, 2, 1]) * scale)
    g = GaussianMixture(4, covariance_type="spherical", init_params="k-means++", random_state=0).fit(rep.reshape(-1, 1))
    o = np.argsort(g.means_[:, 0], kind="stable")
    want_m, want_w = g.means_[o, 0], g.weights_[o]
    assert np.allclose(want_m, [10, 10, 12, 30]) and np.allclose(want_w, [.25, .25, 1 / 3, 1 / 6])
    nq = 64
    got = al.gmm_fit_counts_deep([np.array([10., 12., 30.])] * nq, [np.array([3, 2, 1]) * scale] * nq, 4, None, seed=17)
    assert np.abs(got[:, :4] - want_m).max() < 1e-6
    assert np.abs(got[:, 4:8] - want_w).max() < 1e-6
    assert (got[:, 12] == 4).all()


def _deep_loci(rng, n_loci, A, n_reads=(300, 3000)):
    """Loci of A distinct alleles at least 4 copies apart, +-1 stutter on 6 % of reads, weights normalised."""
    cn, w, rb = [], [], [0]
    for _ in range(n_loci):
        n = int(rng.integers(n_reads[0], n_reads[1] + 1))
        alleles = 8 + 4 * np.sort(rng.choice(np.arange(20), size=A, replace=False)) + rng.integers(0, 2, size=A)
        x = rng.choice(alleles, size=n) + rng.choice([-1, 0, 1], size=n, p=[.03, .94, .03])
        ww = rng.uniform(0.6, 1.4, size=n)
        cn.append(x.astype(np.int32))
        w.append(ww / ww.sum())
        rb.append(rb[-1] + n)
    return np.concatenate(cn), np.concatenate(w), np.asarray(rb, dtype=np.int64)


def _join(parts):
    cn = np.concatenate([p[0] for p in parts])
    w = np.concatenate([p[1] for p in parts])
    rb, off = [np.zeros(1, dtype=np.int64)], 0
    for p in parts:
        rb.append(p[2][1:] + off)
        off += p[2][-1]
    return cn, w, np.concatenate(rb)


def _mixed_batch(rng, n, deep_idx, A, deep_reads=(300, 2000)):
    """n loci with allele counts A; loci deep_idx deep, the rest 8..40 reads."""
    parts = []
    for l in range(n):
        if l in deep_idx:
            parts.append(_deep_loci(rng, 1, min(int(A[l]), 4), deep_reads))
        else:
            parts.append(_poly_loci(rng, 1, 3, n_reads=(8, 40)))
    return _join(parts)


def _without(cn, w, rb, idx):
    """The batch with each locus of idx replaced by a locus of two reads (below min_reads)."""
    parts = []
    for l in range(len(rb) - 1):
        if l in idx:
            parts.append((np.array([20, 21], dtype=np.int32), np.array([.5, .5]), np.array([0, 2], dtype=np.int64)))
        else:
            parts.append((cn[rb[l]:rb[l + 1]], w[rb[l]:rb[l + 1]], np.array([0, rb[l + 1] - rb[l]], dtype=np.int64)))
    return _join(parts)


def test_shallow_rows_unchanged_by_deep_loci_and_deep_rows_are_deterministic(al):
    """1500 loci, A from 1 to 8, 2000 replicates: three chunks of replicate scratch.  60 of the loci are deep.  Every
    shallow row equals, byte for byte, the row of the same batch with each deep locus replaced by one below
    min_reads (same locus indices, S and chunks); deep rows are byte-identical from call to call."""
    rng = np.random.default_rng(515)
    n = 1500
    A = rng.integers(1, 9, size=n).astype(np.int32)
    A[:8] = np.arange(1, 9)
    deep = set(range(8)) | set(int(x) for x in rng.choice(np.arange(8, n), size=52, replace=False))
    cn, w, rb = _mixed_batch(rng, n, deep, A)
    kw = dict(num_bootstrap=2000, seed=31)
    got = al.call_alleles_ploidy_batch(cn, w, rb, A, **kw)
    again = al.call_alleles_ploidy_batch(cn, w, rb, A, **kw)
    ref = al.call_alleles_ploidy_batch(*_without(cn, w, rb, deep), A, **kw)
    d = np.array(sorted(deep))
    s = np.array([l for l in range(n) if l not in deep])
    assert (np.diff(rb)[d] > 256).all() and (np.diff(rb)[s] <= 256).all()
    for x, y in zip(_fields(got, s, 8), _fields(ref, s, 8)):
        assert x.tobytes() == y.tobytes()
    for x, y in zip(_fields(got, d, 8), _fields(again, d, 8)):
        assert x.tobytes() == y.tobytes()
    assert (got.status[d] == 0).all() and (ref.status[d] == 1).all()
    for l in d:
        a = int(A[l])
        xs = cn[rb[l]:rb[l + 1]]
        assert xs.min() <= got.call[l, :a].min() and got.call[l, :a].max() <= xs.max()
        assert np.isclose(got.weights[l, :a].sum(), 1.0) and 1 <= got.modal_n[l] <= a
        assert not got.call[l, a:].any() and not got.means[l, a:].any()
    # the two-allele entry routes the same way
    two = al.call_alleles_batch(cn, w, rb, 2, **kw)
    assert (two.status[d] == 0).all()
    assert (two.call[d] >= 0).all() and np.allclose(two.weights[d].sum(axis=1), 1.0)


def _checker_call(job):
    cn, w, a, seed = job
    return ao.call_alleles(cn, w, a, 4, seed, ao.OracleParams())


def test_deep_calls_agree_with_checker_statistically(al):
    """Tolerance, stated: 60 deep loci (20 each of 2, 3 and 4 alleles, 300-3000 reads, 100 replicates).  The GPU caller
    must agree with the checker (seed set 1) at least as often as the checker agrees with itself under seed set 2,
    minus 8 percentage points for identical calls, 95 % interval bounds within one copy and modal peak counts (one
    locus is 1.7 points); under both checker seeds, no call is more than one copy from the checker's."""
    import multiprocessing as mp
    import os

    rng = np.random.default_rng(3000)
    parts, A = [], []
    for a in (2, 3, 4):
        parts.append(_deep_loci(rng, 20, a))
        A += [a] * 20
    cn, w, rb = _join(parts)
    A = np.array(A, dtype=np.int32)
    ours = al.call_alleles_ploidy_batch(cn, w, rb, A, seed=5)
    assert (ours.status == 0).all()
    with mp.get_context("fork").Pool(min(32, os.cpu_count() or 1)) as pool:
        o1, o2 = ([*pool.map(_checker_call, [(cn[rb[l]:rb[l + 1]], w[rb[l]:rb[l + 1]], int(A[l]), s0 + l)
                                              for l in range(len(A))])] for s0 in (100, 5000))

    def agree(x_call, x_ci, x_modal, y):
        same = np.mean([np.array_equal(x_call[l][:A[l]], y[l]["call"]) for l in range(len(y))])
        ci = np.mean([np.abs(x_ci[l][:A[l]] - y[l]["call_95_cis"]).max() <= 1 for l in range(len(y))])
        modal = np.mean([x_modal[l] == y[l]["modal_n"] for l in range(len(y))])
        return np.array([same, ci, modal])

    self_agree = agree([o["call"] for o in o2], [o["call_95_cis"] for o in o2], [o["modal_n"] for o in o2], o1)
    got_agree = agree(ours.call, ours.call_95_cis, ours.modal_n, o1)
    assert (got_agree >= self_agree - 0.08).all(), (got_agree, self_agree)
    for o in (o1, o2):
        for l in range(len(A)):
            assert np.abs(ours.call[l, :A[l]] - o[l]["call"]).max() <= 1, (l, ours.call[l], o[l]["call"])


def test_edges_256_257_single_value_and_distinct_cap(al):
    rng = np.random.default_rng(257)
    x256 = rng.choice([15, 22], size=256).astype(np.int32)
    x257 = np.concatenate([x256, [15]]).astype(np.int32)
    parts = [(x256, np.full(256, 1 / 256), np.array([0, 256])), (x257, np.full(257, 1 / 257), np.array([0, 257])),
             (np.full(900, 31, dtype=np.int32), np.full(900, 1 / 900), np.array([0, 900])),
             (np.full(300, 12, dtype=np.int32), np.full(300, 1 / 300), np.array([0, 300]))]
    cn, w, rb = _join(parts)
    A = np.array([2, 2, 3, 1], dtype=np.int32)
    r = al.call_alleles_ploidy_batch(cn, w, rb, A, seed=1)
    assert r.status.tolist() == [0, 0, 2, 2]
    assert r.call[0, :2].tolist() == [15, 22] and r.call[1, :2].tolist() == [15, 22]
    assert r.call[2].tolist() == [31, 31, 31] and r.modal_n[2] == 1
    assert np.array_equal(r.weights[2], np.full(3, 1 / 3)) and not r.stdevs[2].any()
    assert r.call_95_cis[2].tolist() == [[31, 31]] * 3 and r.call_99_cis[2].tolist() == [[31, 31]] * 3
    assert r.call[3, 0] == 12 and r.weights[3, 0] == 1.0 and not r.call[3, 1:].any()
    # a deep locus below min_reads: status 1, no call
    r = al.call_alleles_ploidy_batch(cn, w, rb, A, min_reads=600, seed=1)
    assert r.status.tolist() == [1, 1, 2, 1] and not r.call[1].any()
    # over the distinct-value cap
    wide = (np.arange(5000, dtype=np.int32) + 3, np.full(5000, 1 / 5000), np.array([0, 5000]))
    cn2, w2, rb2 = _join(parts[:3] + [wide])
    with pytest.raises(Exception, match="locus 3 has more than 4096 distinct copy numbers"):
        al.call_alleles_ploidy_batch(cn2, w2, rb2, 2)
    ok = (np.arange(4096, dtype=np.int32).repeat(2) + 3, np.full(8192, 1 / 8192), np.array([0, 8192]))
    r = al.call_alleles_ploidy_batch(*_join(parts[:3] + [ok]), 2, num_bootstrap=20)
    assert r.status[3] == 0 and 3 <= r.call[3].min() and r.call[3].max() <= 4098


def test_4096_replicates_eight_alleles_across_chunk_boundaries(al):
    """At A = 8 and 4096 replicates a chunk holds 339 loci; deep loci sit on both sides of the boundaries 339 and 678.
    Their rows do not depend on the chunking or on the other loci: the same batch with every shallow locus replaced
    by one below min_reads gives them byte for byte."""
    rng = np.random.default_rng(4097)
    n = 700
    A = np.full(n, 8, dtype=np.int32)
    deep = {0, 337, 338, 339, 340, 677, 678, 699}
    cn, w, rb = _mixed_batch(rng, n, deep, A, deep_reads=(300, 600))
    got = al.call_alleles_ploidy_batch(cn, w, rb, A, num_bootstrap=4096, seed=8)
    shallow = set(range(n)) - deep
    alone = al.call_alleles_ploidy_batch(*_without(cn, w, rb, shallow), A, num_bootstrap=4096, seed=8)
    d = np.array(sorted(deep))
    assert (got.status[d] == 0).all()
    for x, y in zip(_fields(got, d, 8), _fields(alone, d, 8)):
        assert x.tobytes() == y.tobytes()
    assert ((got.modal_n[d] >= 1) & (got.modal_n[d] <= 8)).all()
    assert np.allclose(got.weights[d].sum(axis=1), 1.0)


def test_drop_in_call_alleles_on_1000_reads(al):
    import types

    params = types.SimpleNamespace(num_bootstrap=100, min_allele_reads=2, force_gm_filter=False,
                                   gmm_params=types.SimpleNamespace(n_init=3, expansion_ratio=5.0, filter_factor=3))
    rng = np.random.default_rng(1000)
    x = rng.choice([18, 26], size=1000)
    fwd, rev = x[:600], x[600:]
    cd = al.call_alleles(fwd, rev, np.full(600, 1e-3), np.full(400, 1e-3), params, 4, 2, False, 0, 42)
    assert isinstance(cd, al.CallData)
    assert cd.call.tolist() == [18, 26] and cd.call_95_cis.shape == (2, 2) and cd.peak_modal_n == 2
    cd4 = al.call_alleles(np.repeat([10, 14, 19, 25], 250), [], np.full(1000, 1e-3), [], params, 4, 4, False, 0, 7)
    assert cd4.call.tolist() == [10, 14, 19, 25]


def test_counting_at_deep_coverage_and_calls_from_the_counts(al):
    """Engine.count_reads on loci of 1000-3000 HiFi-like reads, many of them byte-identical (the dedupe's branch for
    loci of more than 32 reads), bit-exact against the C oracle; the counts then go through the deep allele caller."""
    import strkit_b200
    from strkit_b200 import synth
    from tests import oracle_lib

    oracle = oracle_lib.load()
    params = strkit_b200.RepeatCountParams("repalign", 50, 3, 1)
    eng = strkit_b200.Engine()
    for rpl, n_loci, seed in ((1000, 4, 61), (3000, 2, 62)):
        batch = synth.generate(dataclasses.replace(synth.CONFIGS[2], reads_per_locus=rpl), n_loci, seed=seed).to_host()
        got = eng.count_reads(batch, params)
        want, _ = oracle.count_loci(batch.arena, batch.seq_off, batch.lens, batch.est_cn, batch.read_begin,
                                    batch.motif_off, batch.motif_len, n_threads=8)
        assert np.array_equal(got, want), (rpl, np.flatnonzero((got != want).any(axis=1))[:10])
        st = eng.stats()
        assert st["reads_packed_kernel"] + st["reads_general_kernel"] < 0.8 * batch.n_reads  # identical reads share
        rb = np.asarray(batch.read_begin, dtype=np.int64)
        calls = al.call_alleles_batch(got[:, 0].copy(), np.repeat(1.0 / np.diff(rb), np.diff(rb)), rb, 2, seed=3)
        assert (calls.status != 1).all()
        for l in range(n_loci):
            xs = got[rb[l]:rb[l + 1], 0]
            assert xs.min() <= calls.call[l].min() and calls.call[l].max() <= xs.max()
