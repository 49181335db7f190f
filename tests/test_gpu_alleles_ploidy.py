"""GPU tests of allele calls with per-locus allele counts 1..8 (strk_call_alleles_ploidy, strk_gmm_fit_counts_ploidy)
against the checker (oracle/alleles_oracle.py = numpy + scikit-learn 1.9.0).

What is exact and what is statistical:
  * k-means++ with duplicate centres, EM with k components given the seeds, and fit_gmm's staged filter loop:
    compared with scikit-learn run stage by stage from the same forced seeds, to 1e-6;
  * the aggregation for up to 8 alleles: exact;
  * loci with one or two alleles: byte-identical to strk_call_alleles with the same seed;
  * the whole pipeline draws its own random numbers, so polyploid calls are compared statistically, with the
    tolerance anchored on the checker's own seed-to-seed agreement (stated in the test).
The checker's branches for more than two components (strict filter, staged refit, random fill) restate
allele.py:56-123,249-293; the golden vectors of the reference cover one and two alleles only.
"""
import numpy as np
import pytest

from oracle import alleles_oracle as ao
from tests.alleles_helpers import forced_kmeanspp

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def al():
    import strkit_b200
    from strkit_b200 import alleles

    assert strkit_b200.device_count() > 0, "no CUDA device: these tests need a B200"
    return alleles


def _poly_replicate(rng, A):
    """A sorted replicate with 1..A+1 clusters; some have fewer distinct values than A components."""
    kind = rng.integers(0, 4)
    if kind == 0:  # few distinct values: duplicate centres
        vals = np.sort(rng.choice(np.arange(10, 40), size=int(rng.integers(2, max(3, A))), replace=False))
        x = rng.choice(vals, size=int(rng.integers(A, 40)))
    elif kind == 1:  # A well separated alleles with stutter
        base = np.sort(rng.choice(np.arange(8, 80, 4), size=A, replace=False))
        x = rng.choice(base, size=int(rng.integers(2 * A, 60)))
        x = x + rng.choice([-1, 0, 1], size=x.shape[0], p=[.05, .9, .05])
    elif kind == 2:  # fewer true alleles than A, one lopsided
        k = int(rng.integers(1, A))
        base = np.sort(rng.choice(np.arange(8, 80, 3), size=k, replace=False))
        x = np.concatenate([rng.choice(base, size=int(rng.integers(A, 50))), rng.integers(8, 80, size=int(rng.integers(0, 3)))])
    else:  # noise
        x = rng.integers(10, 40, size=int(rng.integers(A, 80)))
    x = np.sort(x.astype(np.int32), kind="stable")
    if np.unique(x).shape[0] < 2:
        x[-1] += 1
    return x


def _sk_fit(rep, nc, point_seeds):
    from sklearn.mixture import GaussianMixture

    with forced_kmeanspp([point_seeds]):
        return GaussianMixture(n_components=nc, init_params="k-means++", covariance_type="spherical", n_init=1,
                               random_state=0).fit(rep.reshape(-1, 1).astype(np.float64))


def _tie_tol(rep, reg_covar=1e-6):
    """How far apart two restarts' lower bounds may be and still be a tie.  A component that collapses onto one value
    has variance reg_covar, and the log density of its points is the difference of terms of size x^2 / reg_covar that
    cancel: their rounding, eps * x^2 / reg_covar per point, moves the lower bound by several 1e-6 with the order of
    the sums (the mean's last bits differ between any two implementations).  Where that scale is smaller the
    tolerance is 1e-6, as in the two-allele test."""
    return max(1e-6, 16 * 2.220446049250313e-16 * float(np.max(rep)) ** 2 / reg_covar)


def _expected_outcomes(rep, v, c, A, seeds, p, allele_filter):
    """Every acceptable (means, weights, stdevs, peaks, outcome) of fit_gmm on `rep` with the forced seeds: near-tied
    restarts (lower bound within _tie_tol of the best) are followed on every branch of the stages."""
    first_point = np.concatenate([[0], np.cumsum(c)[:-1]])  # a point holding each distinct value
    fits = {}

    def stage_fits(nc):
        if nc not in fits:
            fits[nc] = [_sk_fit(rep, nc, first_point[row]) for row in seeds[nc]]
        return fits[nc]

    out = []

    def single(outcome):
        out.append((np.array([np.mean(rep)]), np.array([1.0]), np.array([np.sqrt(np.var(rep))]), 1, outcome))

    def run(nc, dropped):
        if nc == 1:
            single("single")
            return
        fs = stage_fits(nc)
        best = max(g.lower_bound_ for g in fs)
        for g in fs:
            if g.lower_bound_ < best - _tie_tol(rep):
                continue
            m, w, s = g.means_[:, 0], g.weights_, np.sqrt(g.covariances_)
            useless = ao.count_useless(m, w, nc, allele_filter, p)
            if useless == 0 or nc - useless <= 0:
                o = np.argsort(m, kind="stable")
                outcome = "last_fit" if useless else ("dropped" if dropped else "kept")
                out.append((m[o], w[o], s[o], nc, outcome))
            else:
                run(nc - useless, True)

    run(A, False)
    return out


def _matches_fitted_part(got_row, A, S, want, tol=1e-6):
    """got_row = means[S], weights[S], stdevs[S], n_peaks; the fitted components of `want` must all appear, and every
    entry must be one of them (the fill adds copies drawn at random)."""
    m, w, s, peaks, _ = want
    if int(got_row[3 * S]) != peaks:
        return False
    gm, gw, gs = got_row[:A], got_row[S:S + A], got_row[2 * S:2 * S + A]
    if np.any(got_row[A:S] != 0) or np.any(got_row[S + A:2 * S] != 0) or np.any(got_row[2 * S + A:3 * S] != 0):
        return False
    if np.any(np.diff(gm) < 0):
        return False
    ref = np.stack([m, w, s], axis=1)
    got = np.stack([gm, gw, gs], axis=1)
    close = (np.abs(got[:, None, :] - ref[None, :, :]) / np.maximum(1.0, np.abs(ref[None, :, :])) < tol).all(axis=2)
    if not close.any(axis=1).all():  # an entry that is no fitted component
        return False
    # each fitted component appears at least as often as the fit holds it (duplicate centres give equal components)
    same = (np.abs(ref[:, None, :] - ref[None, :, :]) / np.maximum(1.0, np.abs(ref[None, :, :])) < tol).all(axis=2)
    return bool((close.sum(axis=0) >= same.sum(axis=0)).all())


@pytest.mark.parametrize("A", [3, 4, 5, 6, 7, 8])
def test_staged_fits_match_sklearn_given_the_seeds(al, A):
    """400 replicates per A (100 of them with num_bootstrap = 3, i.e. allele_filter 0.63, which makes fit_gmm drop to a
    single Gaussian or end at <= 0 components and keep its last fit).  Every fit of every stage is scikit-learn from
    the same forced seeds; the GPU row must match one acceptable branch, and all four outcomes must occur."""
    rng = np.random.default_rng(300 + A)
    n_init = 3
    outcomes = set()
    for nb, nq in ((100, 300), (3, 100)):
        p = ao.OracleParams(num_bootstrap=nb)
        allele_filter = (p.min_allele_reads - 0.1) / nb
        values, counts, inits, accept = [], [], [], []
        for q in range(nq):
            rep = _poly_replicate(rng, A)
            v, c = np.unique(rep, return_counts=True)
            seeds = {nc: [rng.choice(len(v), size=nc, replace=len(v) < nc) for _ in range(n_init)]
                     for nc in range(A, 1, -1)}
            accept.append(_expected_outcomes(rep, v, c, A, seeds, p, allele_filter))
            values.append(v.astype(np.float64)), counts.append(c.astype(np.int32))
            inits.append(np.concatenate([np.concatenate(seeds[nc]) for nc in range(A, 1, -1)]))
        got = al.gmm_fit_counts_ploidy(values, counts, A, inits, n_init=n_init, num_bootstrap=nb, seed=A)
        assert got.shape == (nq, 3 * A + 1)
        for q in range(nq):
            ok = [w for w in accept[q] if _matches_fitted_part(got[q], A, A, w)]
            assert ok, (A, nb, q, values[q], counts[q], inits[q], got[q], accept[q])
            outcomes.add(ok[0][4])
    assert outcomes == {"kept", "dropped", "single", "last_fit"}, outcomes


def test_duplicate_centres_from_kmeanspp(al):
    """GaussianMixture(4, spherical, k-means++) on [10, 10, 10, 12, 12, 30]: three centres cover the three values,
    the fourth lands on point 0 (pot = 0), and the two components on 10 stay identical through EM -- whatever the
    random draws.  The GPU's own k-means++ (no forced seeds) must give scikit-learn's result."""
    from sklearn.mixture import GaussianMixture

    rep = np.array([10, 10, 10, 12, 12, 30], dtype=np.float64)
    g = GaussianMixture(4, covariance_type="spherical", init_params="k-means++", random_state=0).fit(rep.reshape(-1, 1))
    o = np.argsort(g.means_[:, 0], kind="stable")
    want_m, want_w = g.means_[o, 0], g.weights_[o]
    assert np.allclose(want_m, [10, 10, 12, 30]) and np.allclose(want_w, [.25, .25, 1 / 3, 1 / 6])
    nq = 256
    got = al.gmm_fit_counts_ploidy([np.array([10., 12., 30.])] * nq, [np.array([3, 2, 1])] * nq, 4, None, seed=17)
    assert np.abs(got[:, :4] - want_m).max() < 1e-6
    assert np.abs(got[:, 4:8] - want_w).max() < 1e-6
    assert (got[:, 12] == 4).all()


def test_aggregation_is_exact_up_to_eight_alleles(al):
    rng = np.random.default_rng(8)
    for A in range(1, 9):
        for B in (3, 100, 1000):
            L = 12
            m = np.round(rng.normal(30, 6, size=(L, A, B)) * 2) / 2  # many ties between replicates
            m.sort(axis=1)
            w = rng.uniform(0.05, 0.9, size=(L, A, B))
            s = rng.uniform(0.0, 2.0, size=(L, A, B))
            peaks = rng.integers(1, A + 1, size=(L, B)).astype(np.uint8)
            if A >= 4 and B == 100:  # ties between several counts: the smallest of the most common wins
                peaks[0] = np.concatenate([np.repeat([A, A - 1, 2], 33), [1]])  # A, A - 1 and 2 tie: 2
                peaks[1] = np.repeat([A, 3], 50)                                 # A and 3 tie: 3
            got = al.aggregate_replicates(m, w, s, peaks)
            for l in range(L):
                want = ao.aggregate(m[l], w[l], s[l], peaks[l])
                assert got.call[l].tolist() == want["call"].tolist()
                assert got.call_95_cis[l].tolist() == want["call_95_cis"].tolist()
                assert got.call_99_cis[l].tolist() == want["call_99_cis"].tolist()
                assert np.array_equal(got.means[l], want["means"]) and np.array_equal(got.stdevs[l], want["stdevs"])
                assert np.allclose(got.weights[l], want["weights"], rtol=0, atol=1e-15)
                assert got.modal_n[l] == want["modal_n"], (A, B, l)


def _poly_loci(rng, n_loci, A, n_reads=(24, 36)):
    """Per-read copy numbers of loci with A alleles (dosage allowed: alleles may repeat), weights normalised."""
    cn, w, rb = [], [], [0]
    for _ in range(n_loci):
        n = int(rng.integers(n_reads[0], n_reads[1] + 1))
        alleles = np.sort(rng.integers(8, 60, size=A))
        x = rng.choice(alleles, size=n) + rng.choice([-1, 0, 1], size=n, p=[.03, .94, .03])
        ww = rng.uniform(0.6, 1.4, size=n)
        cn.append(x.astype(np.int32))
        w.append(ww / ww.sum())
        rb.append(rb[-1] + n)
    return np.concatenate(cn), np.concatenate(w), np.asarray(rb, dtype=np.int64)


def _fields(r, rows, cols):
    return [r.call[rows][:, :cols], r.call_95_cis[rows][:, :cols], r.call_99_cis[rows][:, :cols], r.means[rows][:, :cols],
            r.weights[rows][:, :cols], r.stdevs[rows][:, :cols], r.modal_n[rows], r.status[rows]]


@pytest.mark.parametrize("A", [1, 2])
def test_one_and_two_alleles_are_byte_identical_to_the_uniform_entry(al, A):
    rng = np.random.default_rng(40 + A)
    cn, w, rb = _poly_loci(rng, 400, 2, n_reads=(2, 40))
    old = al.call_alleles_batch(cn, w, rb, A, seed=123)
    new = al.call_alleles_ploidy_batch(cn, w, rb, A, seed=123)
    assert new.call.shape == old.call.shape and (new.n_alleles == A).all()
    for x, y in zip(_fields(old, slice(None), A), _fields(new, slice(None), A)):
        assert x.tobytes() == y.tobytes()


def test_mixed_batch_rows_of_one_and_two_alleles_are_byte_identical(al):
    rng = np.random.default_rng(44)
    n = 600
    A = rng.integers(1, 9, size=n).astype(np.int32)
    cn, w, rb = _poly_loci(rng, n, 3, n_reads=(8, 40))
    new = al.call_alleles_ploidy_batch(cn, w, rb, A, num_bootstrap=200, seed=9)
    assert new.call.shape == (n, 8)
    for a in (1, 2):
        old = al.call_alleles_batch(cn, w, rb, a, num_bootstrap=200, seed=9)
        rows = np.nonzero(A == a)[0]
        assert rows.size > 40
        for x, y in zip(_fields(old, rows, a), _fields(new, rows, a)):
            assert x.tobytes() == y.tobytes()
    for l in range(n):  # unused columns are zero
        assert not new.call[l, A[l]:].any() and not new.means[l, A[l]:].any() and not new.call_95_cis[l, A[l]:].any()
        assert not new.weights[l, A[l]:].any() and not new.stdevs[l, A[l]:].any() and not new.call_99_cis[l, A[l]:].any()
    ok = new.status == 0
    assert np.allclose(new.weights[ok].sum(axis=1), 1.0)
    assert ((new.modal_n[ok] >= 1) & (new.modal_n[ok] <= A[ok])).all()


def _checker_call(job):
    cn, w, a, seed = job
    return ao.call_alleles(cn, w, a, 4, seed, ao.OracleParams())


def test_polyploid_pipeline_agrees_with_checker_statistically(al):
    """Tolerance, stated: over 300 synthetic loci (100 each of 3, 4 and 6 alleles, about 30 reads, 100 replicates), the
    GPU caller must agree with the checker at least as often as the checker agrees with itself under another seed,
    minus 5 percentage points for identical calls and modal peak counts, minus 8 for 95 % interval bounds within one
    copy.  The checker's own interval agreement is only about 0.6 at 5-10 reads per allele (it is about 0.98 for
    the calls), so on 300 loci that rate moves by about 4 points from seed to seed, for the checker too."""
    import multiprocessing as mp
    import os

    rng = np.random.default_rng(2027)
    parts = []
    for A in (3, 4, 6):
        cn, w, rb = _poly_loci(rng, 100, A)
        parts.append((A, cn, w, rb))
    cn = np.concatenate([x[1] for x in parts])
    w = np.concatenate([x[2] for x in parts])
    rb = np.concatenate([[0]] + [x[3][1:] + sum(len(y[1]) for y in parts[:i]) for i, x in enumerate(parts)])
    A = np.concatenate([np.full(100, x[0], dtype=np.int32) for x in parts])
    ours = al.call_alleles_ploidy_batch(cn, w, rb, A, seed=11)
    assert (ours.status == 0).all()

    with mp.get_context("fork").Pool(min(32, os.cpu_count() or 1)) as pool:  # the checker: one process per core
        o1, o2 = ([*pool.map(_checker_call, [(cn[rb[l]:rb[l + 1]], w[rb[l]:rb[l + 1]], int(A[l]), s0 + l)
                                              for l in range(len(A))])] for s0 in (100, 5000))

    def agree(x_call, x_ci, y):
        same = sum(np.array_equal(x_call[l][:A[l]], y[l]["call"]) for l in range(len(y)))
        ci = sum(np.abs(x_ci[l][:A[l]] - y[l]["call_95_cis"]).max() <= 1 for l in range(len(y)))
        return same / len(y), ci / len(y)

    self_same, self_ci = agree([o["call"] for o in o2], [o["call_95_cis"] for o in o2], o1)
    got_same, got_ci = agree(ours.call, ours.call_95_cis, o1)
    assert got_same >= self_same - 0.05, (got_same, self_same)
    assert got_ci >= self_ci - 0.08, (got_ci, self_ci)
    modal_self = np.mean([o2[l]["modal_n"] == o1[l]["modal_n"] for l in range(len(o1))])
    modal_got = np.mean([ours.modal_n[l] == o1[l]["modal_n"] for l in range(len(o1))])
    assert modal_got >= modal_self - 0.05, (modal_got, modal_self)


def test_statuses_and_edges(al):
    """One batch with A = 1..8: empty loci and loci below min_reads (1), single-value loci (2, weights 1/A), fewer
    reads than alleles (3, no call), bootstrapped loci (0)."""
    cn, rb, A = [], [0], []

    def add(x, a):
        cn.extend(x), rb.append(rb[-1] + len(x)), A.append(a)

    for a in range(1, 9):
        add([], a)                                   # empty
        add([12, 13, 14][:min(3, a)], a)             # below min_reads = 4
        add([9] * 7, a)                              # single value
        add([20, 21] * 3 + [20], a)                  # 7 reads: status 3 for a = 8
        add([15, 15, 15, 16, 16, 30, 30, 30] * 2, a)  # 16 reads, bootstrapped
    add([11, 12, 11, 12, 13], 6)                     # 5 reads < 6 alleles: status 3
    cn = np.array(cn, dtype=np.int32)
    rb = np.array(rb, dtype=np.int64)
    A = np.array(A, dtype=np.int32)
    w = np.concatenate([np.full(rb[l + 1] - rb[l], 1.0 / max(1, rb[l + 1] - rb[l])) for l in range(len(A))])
    r = al.call_alleles_ploidy_batch(cn, w, rb, A, seed=3)
    for l in range(len(A)):
        a, n = int(A[l]), int(rb[l + 1] - rb[l])
        xs = cn[rb[l]:rb[l + 1]]
        want = 1 if n < 4 else (2 if np.unique(xs).size == 1 else (3 if n < a else 0))
        assert r.status[l] == want, (l, a, xs, r.status[l])
        if want == 2:
            assert r.call[l, :a].tolist() == [9] * a and r.modal_n[l] == 1
            assert np.array_equal(r.weights[l, :a], np.full(a, 1.0 / a)) and not r.stdevs[l].any()
            assert r.call_95_cis[l, :a].tolist() == [[9, 9]] * a
        if want in (1, 3):
            assert not r.call[l].any() and not r.means[l].any() and r.modal_n[l] == 0
        if want == 0:
            assert xs.min() <= r.call[l, :a].min() and r.call[l, :a].max() <= xs.max() and 1 <= r.modal_n[l] <= a
        assert not r.call[l, a:].any() and not r.weights[l, a:].any()
    for bad in (0, 9):
        A2 = A.copy()
        A2[3] = bad
        with pytest.raises(Exception, match=f"locus 3 has n_alleles = {bad}"):
            al.call_alleles_ploidy_batch(cn, w, rb, A2)


def test_drop_in_raises_the_checker_error_and_calls_polyploid_loci(al):
    import types

    params = types.SimpleNamespace(num_bootstrap=100, min_allele_reads=2, force_gm_filter=False,
                                   gmm_params=types.SimpleNamespace(n_init=3, expansion_ratio=5.0, filter_factor=3))
    cn = np.array([11, 12, 11, 12, 13], dtype=np.int32)
    w = np.full(5, 0.2)
    with pytest.raises(ValueError) as want:
        ao.call_alleles(cn, w, 6, 4, 1, ao.OracleParams())
    with pytest.raises(ValueError) as got:
        al.call_alleles(cn, [], w, [], params, 4, 6, False, 0, 42)
    assert str(got.value) == str(want.value)
    cn3 = np.array([14] * 10 + [17] * 10 + [25] * 10, dtype=np.int32)
    w3 = np.full(30, 1 / 30)
    cd = al.call_alleles(cn3, [], w3, [], params, 4, 3, False, 0, 42)
    assert cd.call.tolist() == [14, 17, 25] and cd.peak_modal_n == 3 and cd.call_95_cis.shape == (3, 2)
    assert al.call_alleles(cn3[:3], [], w3[:3] * 10, [], params, 4, 3, False, 0, 42) is None


def test_chunk_boundaries_at_eight_alleles_and_4096_replicates(al):
    """At A = 8 and 4096 replicates a chunk of replicate scratch holds 339 loci.  Chunk k draws from seed +
    0x9E3779B97F4A7C15 * k with chunk-local locus indices, so each chunk's rows equal a batch of its loci alone."""
    rng = np.random.default_rng(4096)
    n, per = 700, 339
    cn, w, rb = _poly_loci(rng, n, 4, n_reads=(16, 24))
    A = np.full(n, 8, dtype=np.int32)
    A[::5] = 2  # the stride stays 8: per-locus counts below the maximum do not move the chunk boundaries
    seed = 77
    whole = al.call_alleles_ploidy_batch(cn, w, rb, A, num_bootstrap=4096, seed=seed)
    assert (whole.status == 0).all()
    for k, l0 in enumerate(range(0, n, per)):
        l1 = min(n, l0 + per)
        part = al.call_alleles_ploidy_batch(cn[rb[l0]:rb[l1]], w[rb[l0]:rb[l1]], rb[l0:l1 + 1] - rb[l0], A[l0:l1],
                                            num_bootstrap=4096, seed=(seed + 0x9E3779B97F4A7C15 * k) & (2**64 - 1))
        for x, y in zip(_fields(whole, slice(l0, l1), 8), _fields(part, slice(None), 8)):
            assert x.tobytes() == y.tobytes(), k
