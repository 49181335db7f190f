"""strk_ref_counts (get_ref_repeat_count for a batch of loci) against the CPU oracle, row by row, on the calls that
reach past its device-resident part: several search-parameter tiers in one call, respect_coords, more searches out of
their first window than the second look takes, windows too wide for the packed kernel, a matrix the packed kernel
cannot take, and max_iters = 0."""
from __future__ import annotations

import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from strkit_b200.align_matrix import dna_matrix
from tests.helpers import families_to_batch, mutate, rand_seq
from tests.oracle_lib import GAP, Oracle

pytestmark = pytest.mark.gpu

# repeat_count_params.py:17-42, (max_iters, local search range, step size): below 200, from 200, 1000, 2000 copies
TIERS = [(250, 3, 1), (200, 3, 3), (150, 3, 5), (50, 1, 15)]


@pytest.fixture(scope="module")
def sb():
    import strkit_b200

    assert strkit_b200.device_count() > 0, "no CUDA device: these tests must run on the GPU box"
    return strkit_b200


@pytest.fixture(scope="module")
def pool():
    # the oracle's ctypes calls release the GIL
    with ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 4)) as ex:
        yield ex


def make_loci(seed, n, k_range=(5, 60), shift=None, shifted=0.2):
    """n reference windows (motif, tract, flank, flank) and start counts; a `shifted` share of the start counts moved by
    rng.integers(*shift) copies, so that their searches leave the first window."""
    rng = np.random.default_rng(seed)
    fams, starts = [], []
    for i in range(n):
        m = int(rng.integers(2, 7))
        motif = rand_seq(rng, m)
        tr = mutate(rng, motif * int(rng.integers(*k_range)), 0.01, 0.005, 0.005)
        fl, fr = rand_seq(rng, 70), rand_seq(rng, 70)
        if i % 3 == 0:  # the repeat spills into the flanks: phase 1 moves the boundaries
            fl = fl[:60] + (motif * 10)[-10:]
            fr = (motif * 10)[:8] + fr[8:]
        fams.append((motif, tr, fl, fr))
        starts.append(round(len(tr) / m))
    starts = np.array(starts, dtype=np.int32)
    if shift is not None:
        moved = rng.random(n) < shifted
        starts[moved] = np.maximum(0, starts[moved] + rng.integers(*shift, int(moved.sum())))
    return fams, starts


def check(sb, oracle, pool, fams, starts, rcs, respect_coords=False, matrix=None):
    """One strk_ref_counts call; every row must equal the oracle's (the same matrix).  Returns the call's counters."""
    eng = sb.Engine() if matrix is None else sb.Engine(matrix=matrix)
    sizes = [len(f[1]) for f in fams]
    got = eng.ref_counts(families_to_batch(fams), starts, sizes, np.array(rcs, dtype=np.int32), vcf_anchor_size=5,
                         respect_coords=respect_coords)
    st = eng.stats()
    eng.close()

    def want(i):
        motif, tr, fl, fr = fams[i]
        (cn, score), lo, ro, (n_off, n_fin), (fl2, _, fr2) = oracle.get_ref_repeat_count(
            int(starts[i]), tr, fl, fr, motif, sizes[i], 5, *rcs[i], respect_coords=respect_coords)
        return [cn, score, lo, ro, n_off, n_fin, len(fl2), len(fr2)]

    rows = list(pool.map(want, range(len(fams))))
    bad = [i for i, row in enumerate(rows) if got[i].tolist() != row]
    assert not bad, [(i, fams[i][0], rcs[i], int(starts[i]), got[i].tolist(), rows[i]) for i in bad[:5]]
    return st


def test_mixed_tiers_and_bad_starts(sb, oracle, pool):
    """All four tiers in one call, a fifth of the start counts off by tens of copies: phase 1's second look and the
    host finish both run inside a multi-tier call."""
    fams, starts = make_loci(31, 400, k_range=(5, 120), shift=(-40, 80))
    st = check(sb, oracle, pool, fams, starts, [TIERS[i % 4] for i in range(len(fams))])
    assert st["widening_passes"] > 0   # loci finished on the host


def test_respect_coords_mixed_tiers(sb, oracle, pool):
    """respect_coords (no boundary search) on a batch of every tier; shifted starts send phase 2 past its window."""
    fams, starts = make_loci(32, 160, k_range=(5, 120), shift=(-30, 60))
    check(sb, oracle, pool, fams, starts, [TIERS[(i * 7) % 4] for i in range(len(fams))], respect_coords=True)


def test_past_the_second_look_cap(sb, oracle, pool):
    """One tier, 5000 loci nearly all started 8-20 copies off: more than the second look's 4096 loci leave the first
    window (+-6 sizes), and the host finishes the ones beyond the cap."""
    fams, starts = make_loci(33, 5000, k_range=(25, 60), shift=(8, 21), shifted=0.97)
    down = np.random.default_rng(34).random(len(fams)) < 0.5   # half of the moves downwards
    base = np.array([round(len(f[1]) / len(f[0])) for f in fams], dtype=np.int32)
    starts = np.where(down, np.maximum(0, 2 * base - starts), starts).astype(np.int32)
    st = check(sb, oracle, pool, fams, starts, [TIERS[0]] * len(fams))
    assert st["widening_passes"] > len(fams) - 4096   # at least the loci beyond the cap were finished on the host


@pytest.mark.parametrize("wide", [(100, 10, 25), (100, 30, 40)], ids=["phase1_window", "phase2_window"])
def test_windows_too_wide_for_packed(sb, oracle, pool, wide):
    """A tier whose first boundary window (range + step + 2 > 31 sizes either side: forward and reverse columns pass
    PK_WINDOW_MAX) or whose phase 2 window (> 63 either side) is too wide for the packed kernel, next to a normal tier."""
    fams, starts = make_loci(35 + wide[1], 120, shift=(-20, 40))
    check(sb, oracle, pool, fams, starts, [wide if i % 2 else TIERS[0] for i in range(len(fams))])


@pytest.mark.parametrize("tiers", [1, 4])
def test_matrix_not_packed_ok(sb, oracle, pool, tiers):
    """A matrix with one entry below -2g: the packed kernel cannot hold its scores, every DP runs on the general kernel;
    against an oracle that uses the same matrix."""
    mat = dna_matrix.astype(np.int16).copy()
    mat[0, 1] = mat[1, 0] = -2 * GAP - 1
    mat = mat.astype(np.int8)
    o = Oracle(oracle.lib)
    o.matrix = np.ascontiguousarray(mat.reshape(-1), dtype=np.int8)
    fams, starts = make_loci(36, 120, shift=(-20, 40))
    check(sb, o, pool, fams, starts, [TIERS[i % tiers] for i in range(len(fams))], matrix=mat)


@pytest.mark.parametrize("tiers", [1, 4])
def test_max_iters_zero(sb, tiers):
    """max_iters = 0 scores no size: the call fails with the first such locus, in a one-tier and a multi-tier call."""
    from strkit_b200._native import StrkError

    fams, starts = make_loci(37, 12)
    rcs = [(0, 3, 1) if tiers == 1 or i % 4 == 1 else TIERS[i % 4] for i in range(len(fams))]
    first = 0 if tiers == 1 else 1
    eng = sb.Engine()
    with pytest.raises(StrkError, match=rf"strk_ref_counts: locus {first} scored no size \(max_iters = 0\)"):
        eng.ref_counts(families_to_batch(fams), starts, [len(f[1]) for f in fams], np.array(rcs, dtype=np.int32), 5)
    eng.close()
