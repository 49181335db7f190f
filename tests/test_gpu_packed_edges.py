"""Edges of the packed u16x2 kernel (dp_packed.cuh), entry by entry against the CPU oracle.

Every table below is compared with the oracle entry by entry, and every call predicts how many families the packed
kernel keeps: a family that silently falls back to the general kernel computes the right numbers, so only the
routing assertion shows that the packed code was the one tested.  The inputs sit where the packed kernel goes wrong
quietly: reference-mode tables (score and smallest row per size), windows of up to PK_WINDOW_MAX sizes (the later
rounds of the combine), two reads per warp that differ in every shared quantity, both sides of the class, flank,
motif and 16-bit range gates, matrices whose PRMT byte lanes all differ, and work lists longer than the resident
warps."""
from __future__ import annotations

import os
from collections import defaultdict
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from strkit_b200.align_matrix import dna_matrix
from strkit_b200.batcher import LocusReads, ReadBatch, pack_loci
from tests.helpers import families_to_batch, rand_seq
from tests.oracle_lib import GAP, Oracle

pytestmark = pytest.mark.gpu

# restated from strkit_b200/csrc/dp_packed.cuh:48-49 and strk_common.cuh:77
PK_FLANK_MAX = 160
PK_WINDOW_MAX = 128
PK_RMAX = 16
PK_PAIR_RMAX = 8        # api.cu:577: classes up to 8 run two reads per warp (16 lanes each)
IUPAC_ONLY = set("RYSWKMBDHVryswkmbdhv")   # row symbols the packed kernel has no PRMT class for (api.cu:283, 301)


@pytest.fixture(scope="module")
def sb():
    import strkit_b200

    assert strkit_b200.device_count() > 0, "no CUDA device: these tests must run on the GPU box"
    return strkit_b200


@pytest.fixture(scope="module")
def pool():
    # the oracle's ctypes calls release the GIL: the scalar alignments of one table run on every core
    with ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 4)) as ex:
        yield ex


# ------------------------------------------------------------------------------------------------ routing model
def pk_class(fl: int, tr: int, fr: int, m: int) -> int:
    """strk_pk_class (plan.cuh:30-34) with strk_pick_rows_packed (strk_common.cuh:79-83): rows per lane, 0 = general."""
    r = max(2, (fl + tr + fr + 1 + 31) // 32)
    if r > PK_RMAX:
        return 0
    if fl < 1 or fr < 1 or fl > PK_FLANK_MAX or fr > PK_FLANK_MAX or m * r > 128 or m <= 0:
        return 0
    return r


def pk_ncols(fl: int, fr: int, m: int, n_lo: int, n_hi: int, ref: bool) -> int:
    """Columns the longer half sweeps: the split b0 and ncols of dp_packed.cuh:419-427."""
    if ref:  # both halves sweep the whole prefix chain
        return max(fl, fr) + m * n_hi
    num = m * n_hi + fl - fr + m
    b0 = num // (2 * m) if num >= 0 else -(-num // (2 * m))   # C division truncates toward zero
    b0 = min(max(b0, 0), n_lo)
    return max(fl + m * (n_hi - b0), fr + m * b0)


def pk_range_ok(fl: int, tr: int, fr: int, m: int, n_lo: int, n_hi: int, ref: bool) -> bool:
    """The u16 range gate of dp_packed.cuh:434 with g = 5 and N = 32 R rows (both lane counts: 16 lanes x 2R rows)."""
    n = 32 * pk_class(fl, tr, fr, m)
    return GAP * (n + pk_ncols(fl, fr, m, n_lo, n_hi, ref) + 40) + 2 * n + 1024 < (32000 if ref else 65535)


def table_class(fam, lo: int, hi: int, ref: bool) -> int:
    """tables_common (api.cu): the batch paths' window rule on top of the class rule."""
    motif, tr, fl, fr = fam
    w = hi - lo + 1
    if (2 * w if ref else w) > PK_WINDOW_MAX:
        return 0
    return pk_class(len(fl), len(tr), len(fr), len(motif))


def predict_packed(fams, n_lo, n_hi, ref: bool) -> int:
    return len(packed_set(fams, n_lo, n_hi, ref))


def packed_set(fams, n_lo, n_hi, ref: bool) -> set:
    """Indices of the families the packed kernel keeps.  A class list holds its families in input order; with 16 lanes a warp sweeps
    list items 2j and 2j + 1 and hands both to the general kernel when either one is ineligible (dp_packed.cuh:431-439,
    496-499).  A last odd item re-runs in the idle unit, so it pairs with itself."""
    lists = defaultdict(list)
    for i, (f, lo, hi) in enumerate(zip(fams, n_lo, n_hi)):
        k = table_class(f, int(lo), int(hi), ref)
        if k:
            lists[k].append(i)

    def eligible(i):
        motif, tr, fl, fr = fams[i]
        return (not (set(fl + tr + fr) & IUPAC_ONLY) and
                pk_range_ok(len(fl), len(tr), len(fr), len(motif), int(n_lo[i]), int(n_hi[i]), ref))

    kept = set()
    for k, items in lists.items():
        per = 2 if k <= PK_PAIR_RMAX else 1
        for j in range(0, len(items), per):
            unit = items[j:j + per]
            if all(eligible(i) for i in unit):
                kept.update(unit)
    return kept


def test_routing_model_restates_the_gates():
    """The model itself, on hand-worked cases."""
    assert [pk_class(1, 30, 0, 1), pk_class(1, 29, 1, 1), pk_class(1, 30, 1, 1)] == [0, 2, 2]
    assert [pk_class(10, 43, 10, 2), pk_class(10, 44, 10, 2)] == [2, 3]
    assert [pk_class(100, 311, 100, 8), pk_class(100, 312, 100, 8)] == [16, 0]
    assert [pk_class(160, 10, 5, 1), pk_class(161, 10, 5, 1)] == [6, 0]
    assert [pk_class(10, 20, 10, 64), pk_class(10, 20, 10, 65), pk_class(200, 300, 11, 8), pk_class(200, 300, 11, 9)] \
        == [2, 0, 0, 0]
    assert [pk_class(100, 300, 100, 8), pk_class(100, 300, 100, 9)] == [16, 0]
    # read mode, R = 2: 5 * (64 + 12772 + 40) + 128 + 1024 = 65532 < 65535, one more column is 65537
    assert (gate_limit(2, False), gate_limit(16, False), gate_limit(2, True)) == (12772, 12145, 6065)
    assert pk_ncols(20, 20, 1, 25000, 25000, False) == 12520 and pk_ncols(7, 3, 5, 10, 12, True) == 67
    assert pk_ncols(3, 90, 4, 0, 5, False) == 90 and pk_ncols(90, 3, 4, 30, 31, False) == 90 + 4 * 5
    assert pk_range_ok(20, 20, 20, 1, 25000, 25000, False) and not pk_range_ok(20, 20, 20, 1, 25000, 25506, False)


# ------------------------------------------------------------------------------------------------ families
def periodic(rng, motif: str, n: int, sub: float = 0.03) -> str:
    """n bases of the motif's repeat (IUPAC codes drawn as a concrete base), with substitutions only: exact length."""
    if n <= 0:
        return ""
    conc = [c if c in "ACGT" else str(rng.choice(list("ACGT"))) for c in motif.upper()]
    s = [conc[i % len(conc)] for i in range(n)]
    for i in np.flatnonzero(rng.random(n) < sub):
        s[i] = str(rng.choice(list("ACGT")))
    return "".join(s)


def make_family(rng, n1: int, m: int, fl: int, fr: int, variant: int):
    """A family of exactly n1 = fl + tr + fr bases and a motif of m bases.  variant: 0 plain, 1 homopolymer and
    2 dinucleotide tracts that run into both flanks (tie-heavy), 3 N / X rows, 4 lower case, 5 an IUPAC motif."""
    tr_len = n1 - fl - fr
    assert tr_len >= 0, (n1, fl, fr)
    if variant == 1:
        m = 1
        motif = "A"
    elif variant == 2 and m >= 2:
        m = 2
        motif = "AC"
    else:
        motif = rand_seq(rng, m)
    if variant == 5:
        motif = "".join(str(rng.choice(list("RYN"))) if j % 3 == 1 else c for j, c in enumerate(motif))
    tr = periodic(rng, motif, tr_len, 0.0 if variant in (1, 2) else 0.03)
    fls, frs = rand_seq(rng, fl), rand_seq(rng, fr)
    if variant in (1, 2):  # the repeat continues into the flanks
        run = (motif * 8)[: min(6, fl)]
        fls = fls[: fl - len(run)] + run
        run = (motif * 8)[: min(6, fr)]
        frs = run + frs[len(run):]
    if variant == 3:
        noisy = lambda s: "".join("N" if u < 0.04 else ("X" if u < 0.1 else c) for c, u in zip(s, rng.random(len(s))))  # noqa: E731
        tr, fls, frs = noisy(tr), noisy(fls), noisy(frs)
    if variant == 4:
        tr, fls = tr.lower(), fls.lower()
    return (motif, tr, fls, frs)


def window(fam, w: int, lo_min: int = 0, zero: bool = False):
    motif, tr = fam[0], fam[1]
    if zero:
        return 0, w - 1
    est = round(len(tr) / len(motif))
    lo = max(lo_min, est - w // 2)
    return lo, lo + w - 1


def class_family(rng, R: int, variant: int, m_max: int = 8, flank_max: int = 70):
    """A family of class R (n1 in [32(R-1), 32R-1], m * R <= 128)."""
    n1 = int(rng.integers(max(3, 32 * (R - 1)), 32 * R))
    m = int(rng.integers(1, min(m_max, 128 // R) + 1))
    f_cap = max(1, min(flank_max, (n1 - 1) // 2))
    fl, fr = int(rng.integers(1, f_cap + 1)), int(rng.integers(1, f_cap + 1))
    fam = make_family(rng, n1, m, fl, fr, variant)
    assert pk_class(len(fam[2]), len(fam[1]), len(fam[3]), len(fam[0])) == R
    return fam


# ------------------------------------------------------------------------------------------------ checks
def oracle_read_tables(oracle, pool, fams, n_lo, n_hi, flags):
    def one(args):
        (motif, tr, fl, fr), lo, hi = args
        return [oracle.score_candidate(tr, fl, fr, motif, n, flags) for n in range(lo, hi + 1)]

    rows = pool.map(one, zip(fams, (int(v) for v in n_lo), (int(v) for v in n_hi)))
    return np.asarray([v for r in rows for v in r], dtype=np.int32)


def oracle_ref_tables(oracle, pool, fams, n_lo, n_hi):
    """(fwd_score, fwd r_adj, rev_score, rev l_adj) per size: end_query as score_ref_boundaries uses it."""
    def one(args):
        (motif, tr, fl, fr), lo, hi = args
        out = []
        for n in range(lo, hi + 1):
            (fs, ra), (rs, la) = oracle.score_ref_boundaries(tr, fl, fr, motif, n, len(tr))
            out.append((fs, ra, rs, la))
        return out

    rows = pool.map(one, zip(fams, (int(v) for v in n_lo), (int(v) for v in n_hi)))
    return np.asarray([v for r in rows for v in r], dtype=np.int32).reshape(-1, 4)


def ref_adjusted(tab, fams, n_lo, n_hi):
    """The device's end_query turned into score_ref_boundaries' adjusted offsets (repeats.py:34,41)."""
    adj = tab.copy()
    k = 0
    for (motif, tr, fl, fr), lo, hi in zip(fams, n_lo, n_hi):
        w = int(hi) - int(lo) + 1
        adj[k:k + w, 1] += 1 - len(fl) - len(tr)
        adj[k:k + w, 3] += 1 - len(fr) - len(tr)
        k += w
    return adj


def first_bad(got, want, fams, n_lo, n_hi):
    """Which family and size the first differing entry belongs to (for the assertion message)."""
    bad = np.flatnonzero((got != want).reshape(got.shape[0], -1).any(axis=1)) if got.shape == want.shape else [0]
    if len(bad) == 0:
        return None
    widths = np.asarray(n_hi, dtype=np.int64) - np.asarray(n_lo, dtype=np.int64) + 1
    fi = int(np.searchsorted(np.cumsum(widths), bad[0], side="right"))
    motif, tr, fl, fr = fams[fi]
    return dict(entry=int(bad[0]), n_bad=len(bad), family=fi, n=int(n_lo[fi]) + int(bad[0] - (np.cumsum(widths)[fi] - widths[fi])),
                motif=motif, lens=(len(fl), len(tr), len(fr)), window=(int(n_lo[fi]), int(n_hi[fi])),
                got=got[bad[0]].tolist(), want=want[bad[0]].tolist())


def check_read(sb, oracle, pool, fams, n_lo, n_hi, flags=15, matrix=None, general=True):
    n_lo, n_hi = np.asarray(n_lo, dtype=np.int32), np.asarray(n_hi, dtype=np.int32)
    eng = sb.Engine(end_flags=flags) if matrix is None else sb.Engine(end_flags=flags, matrix=matrix)
    batch = families_to_batch(fams)
    got, _ = eng.score_tables(batch, n_lo, n_hi)
    st = eng.stats()
    want = oracle_read_tables(oracle, pool, fams, n_lo, n_hi, flags)
    assert np.array_equal(got, want), first_bad(got, want, fams, n_lo, n_hi)
    kept = predict_packed(fams, n_lo, n_hi, ref=False)
    assert (st["reads_packed_kernel"], st["reads_general_kernel"]) == (kept, len(fams) - kept)
    if general:
        again, _ = eng.score_tables(batch, n_lo, n_hi, kernel=sb.KERNEL_GENERAL)
        assert np.array_equal(again, want) and eng.stats()["reads_packed_kernel"] == 0
    eng.close()
    return kept


def check_ref(sb, oracle, pool, fams, n_lo, n_hi, matrix=None, general=True):
    n_lo, n_hi = np.asarray(n_lo, dtype=np.int32), np.asarray(n_hi, dtype=np.int32)
    eng = sb.Engine() if matrix is None else sb.Engine(matrix=matrix)
    batch = families_to_batch(fams)
    tab, _ = eng.ref_boundary_tables(batch, n_lo, n_hi)
    st = eng.stats()
    want = oracle_ref_tables(oracle, pool, fams, n_lo, n_hi)
    got = ref_adjusted(tab, fams, n_lo, n_hi)
    assert np.array_equal(got, want), first_bad(got, want, fams, n_lo, n_hi)
    kept = predict_packed(fams, n_lo, n_hi, ref=True)
    assert (st["reads_packed_kernel"], st["reads_general_kernel"]) == (kept, len(fams) - kept)
    if general:
        again, _ = eng.ref_boundary_tables(batch, n_lo, n_hi, kernel=sb.KERNEL_GENERAL)
        assert np.array_equal(again, tab) and eng.stats()["reads_packed_kernel"] == 0
    eng.close()
    return kept


# ------------------------------------------------------------------------------------------------ 1. reference mode
REF_WIDTHS = (1, 2, 3, 4, 5, 13, 31, 32, 63, 64)


def ref_class_families(R: int, seed: int):
    rng = np.random.default_rng(seed)
    fams, lo, hi = [], [], []
    for j, w in enumerate(REF_WIDTHS + (65,)):
        for v in range(3):
            variant = (j + 2 * v) % 6
            fam = class_family(rng, R, variant)
            a, b = window(fam, w, zero=(v == 2 and j % 2 == 0))
            fams.append(fam), lo.append(a), hi.append(b)
    return fams, lo, hi


@pytest.mark.parametrize("R", range(2, PK_RMAX + 1))
def test_ref_tables_packed_every_class(sb, oracle, pool, R):
    """Reference windows of every class, both lane counts, W up to 64 (2W <= PK_WINDOW_MAX) and 65 (general kernel):
    (score, end_query) of both directions at every size against score_ref_boundaries.  Homopolymer and dinucleotide
    tracts that run into the flanks put the column maximum on several rows (only the smallest is parasail's)."""
    fams, lo, hi = ref_class_families(R, 1000 + R)
    kept = check_ref(sb, oracle, pool, fams, lo, hi)
    assert kept == len(fams) - 3   # all but the three 65-size windows


# ------------------------------------------------------------------------------------------------ 2. read-mode widths
READ_WIDTHS = tuple(range(1, 10)) + (15, 16, 17, 31, 32, 33, 63, 64, 65, 127, 128)
READ_CLASSES = (2, 5, 8, 9, 12, 16)


def read_width_families(seed: int, classes=READ_CLASSES, widths=READ_WIDTHS + (129,)):
    rng = np.random.default_rng(seed)
    fams, lo, hi = [], [], []
    for R in classes:
        for j, w in enumerate(widths):
            fam = class_family(rng, R, j % 6)
            a, b = window(fam, w, zero=(j % 7 == 3))
            fams.append(fam), lo.append(a), hi.append(b)
    return fams, lo, hi


@pytest.mark.parametrize("flags", [0, 2, 4, 5, 8, 10, 12, 15])
def test_read_tables_window_widths(sb, oracle, pool, flags):
    """Windows of 1..128 sizes in classes of both lane counts: every round of the combine's L-candidate loop and
    every remainder of its batches of 4; the end flags reach the last-row prefix maximum (s2_end) and the backward
    border (s2_beg) of the close.  W = 129 goes to the general kernel."""
    fams, lo, hi = read_width_families(2000 + flags)
    kept = check_read(sb, oracle, pool, fams, lo, hi, flags)
    assert kept == len(fams) - len(READ_CLASSES)   # every family but the 129-size windows


# ------------------------------------------------------------------------------------------------ 3. paired warps
def paired_families(seed: int, ref: bool):
    """Pairs of class-6 families (16 lanes, two reads per warp) that differ in one shared quantity each; every pair
    also appears in the other order, so each member runs in both halves of a warp."""
    rng = np.random.default_rng(seed)
    w_big = 64 if ref else 128

    def fam(fl=20, fr=20, n1=176, m=4, variant=0):
        return make_family(rng, n1, m, fl, fr, variant)

    pairs = []
    a, b = fam(), fam()
    pairs.append(((a,) + window(a, 1), (b,) + window(b, w_big)))                    # window 1 with window 128 (64)
    a, b = fam(fl=1, fr=30, m=5), fam(fl=160, fr=3, m=7)
    pairs.append(((a,) + window(a, 9), (b,) + window(b, 9)))                       # union Lmax, mid-motif phase
    a, b = fam(), fam(variant=3)
    pairs.append(((a,) + window(a, 6), (b,) + window(b, 6)))                       # plain rows with N / X rows
    a, b = fam(m=6), fam(m=6, variant=5)
    pairs.append(((a,) + window(a, 5), (b,) + window(b, 5)))                       # ACGT motif with IUPAC motif
    a, b = fam(m=3), fam(m=1, fl=10, fr=10)
    pairs.append(((a,) + window(a, 7, zero=True), (b,) + window(b, 7)))            # n_lo = 0 with n_lo ~ 150
    a, b = fam(), fam()
    b = (b[0], b[1][:40] + "R" + b[1][41:], b[2], b[3])
    pairs.append(((a,) + window(a, 4), (b,) + window(b, 4)))                       # IUPAC inside one read: both fall back
    a, b = fam(), fam(m=20, fl=10, fr=10, n1=170)
    far = 1280 if not ref else 300                                                 # ~ 12 600 / 6 000 columns
    assert not pk_range_ok(10, 150, 10, 20, far - 1, far, ref)
    pairs.append(((a,) + window(a, 3), (b, far - 1, far)))                         # range gate fails for one read
    fams, lo, hi = [], [], []
    for x, y in pairs:
        for f, l, h in (x, y, y, x):
            fams.append(f), lo.append(l), hi.append(h)
    a = fam()
    for f, l, h in ((a,) + window(a, 5),):                                         # odd list: a unit without a read
        fams.append(f), lo.append(l), hi.append(h)
    assert {pk_class(len(f[2]), len(f[1]), len(f[3]), len(f[0])) for f in fams} == {6}
    return fams, lo, hi


@pytest.mark.parametrize("mode", ["read", "ref"])
def test_paired_warps_mismatched_units(sb, oracle, pool, mode):
    fams, lo, hi = paired_families(3000, mode == "ref")
    if mode == "read":
        kept = check_read(sb, oracle, pool, fams, lo, hi, 15)
    else:
        kept = check_ref(sb, oracle, pool, fams, lo, hi)
    assert kept == len(fams) - 8   # the IUPAC pair and the range-gate pair, in both orders


# ------------------------------------------------------------------------------------------------ 4. gates
def gate_family(rng, R: int, target: int, ref: bool, w: int = 2):
    """A class-R family with a long motif whose longer half sweeps exactly `target` columns (pk_ncols)."""
    n1 = 32 * R - 20
    for m in range(128 // R, 0, -1):
        for fl in range(1, min(PK_FLANK_MAX, n1 // 2) + 1):
            fr = fl
            for n_hi in range(max(w, (target - fl) // m - 2), target // max(1, m // 2) + 3):
                if pk_ncols(fl, fr, m, n_hi - w + 1, n_hi, ref) == target:
                    fam = make_family(rng, n1, m, fl, fr, 0)
                    assert pk_class(fl, len(fam[1]), fr, m) == R
                    return fam, n_hi - w + 1, n_hi
    raise AssertionError(f"no family of class {R} sweeps {target} columns")


def gate_limit(R: int, ref: bool) -> int:
    """Largest ncols the range gate lets through for class R."""
    n = 32 * R
    lim = 32000 if ref else 65535
    return (lim - 1 - 2 * n - 1024) // GAP - n - 40


def edge_families(seed: int, ref: bool):
    rng = np.random.default_rng(seed)
    fams, lo, hi = [], [], []

    def add(fam, a, b):
        fams.append(fam), lo.append(a), hi.append(b)

    for R in range(2, PK_RMAX + 1):          # n1 = 32(R-1): 32 pad rows; 32R - 1: one pad row
        for n1 in (32 * (R - 1), 32 * R - 1):
            f = make_family(rng, n1, 2, min(30, n1 // 3), min(25, n1 // 3), R % 4)
            add(f, *window(f, 3 + R % 3, lo_min=1))
    for n1 in (3, 4, 5):                     # tiny reads in R = 2
        f = make_family(rng, n1, 1, 1, 1, 0)
        add(f, *window(f, 3, lo_min=1))
    f = make_family(rng, 512, 4, 60, 60, 0)  # 512 bases: the general kernel
    add(f, *window(f, 3, lo_min=1))
    for fl in (0, 1, 160, 161):              # flank gates
        for fr in (0, 1, 160, 161):
            f = make_family(rng, fl + fr + 40, 4, fl, fr, (fl + fr) % 4)
            add(f, *window(f, 3, lo_min=1))
    for R, m in ((2, 64), (2, 65), (16, 8), (16, 9)):   # m * R = 128 / 129
        f = make_family(rng, 32 * R - 10, m, 3, 3, 0)
        add(f, *window(f, 2, lo_min=1))
    gates = []
    for R in (2, 16) if not ref else (2,):  # range gate: one column inside, one outside, one far outside
        lim = gate_limit(R, ref)
        # far: g * (N + ncols) > 70 000, so the biased cells of the longer half really pass 16 bits
        for target, ok in ((lim, True), (lim + 1, False), (14100 - 32 * R, False)):
            gates.append((len(fams), ok))
            add(*gate_family(rng, R, target, ref, w=1 + target % 4))
    return fams, lo, hi, gates


@pytest.mark.parametrize("mode", ["read", "ref"])
def test_class_and_gate_edges(sb, oracle, pool, mode):
    """Both sides of every gate of the packed kernel, with the kernel that ran asserted through the routing model:
    class boundaries (one and 32 pad rows, 511 / 512 bases), flanks 0 / 1 / 160 / 161, m * R = 128 / 129, and the
    u16 range gate one column inside, one outside and far enough outside that biased cells pass 16 bits."""
    ref = mode == "ref"
    fams, lo, hi, gates = edge_families(4000 + ref, ref)
    packed = packed_set(fams, lo, hi, ref)
    assert {pk_class(len(fams[i][2]), len(fams[i][1]), len(fams[i][3]), len(fams[i][0])) for i in packed} == \
        set(range(2, PK_RMAX + 1))   # with the routing assertion: the packed kernel ran every class
    for i, ok in gates:   # the family just inside runs on the packed kernel, the ones outside do not
        motif, tr, fl, fr = fams[i]
        assert pk_range_ok(len(fl), len(tr), len(fr), len(motif), lo[i], hi[i], ref) is ok and (i in packed) is ok
    if ref:
        kept = check_ref(sb, oracle, pool, fams, lo, hi)
    else:
        kept = check_read(sb, oracle, pool, fams, lo, hi, 15)
    assert kept >= 2 * (PK_RMAX - 1)


# ------------------------------------------------------------------------------------------------ 5. matrices
def _sym(mat, a, b, v):
    mat[a, b] = mat[b, a] = v


def matrix_m1() -> np.ndarray:
    """Symmetric, every N / X / other row constant over A/C/G/T (one_table_ok = 1), but the byte lanes all differ:
    a match score per base, transitions apart from transversions, N, X and "other" rows of their own."""
    mat = dna_matrix.astype(np.int16).copy()
    acgt = [[3, -6, -2, -5], [-6, 2, -4, -3], [-2, -4, 4, -6], [-5, -3, -6, 1]]
    mat[:4, :4] = acgt
    for b in range(4):
        _sym(mat, 14, b, -1)    # N
        _sym(mat, 15, b, 0)     # X
        _sym(mat, 16, b, -3)    # other
    _sym(mat, 14, 15, -2)
    _sym(mat, 14, 16, 1)
    _sym(mat, 15, 16, -4)
    mat[14, 14], mat[15, 15], mat[16, 16] = 1, 2, -1
    return mat.astype(np.int8)


def matrix_m2() -> np.ndarray:
    """M1 with an X row that scores differently against each base: one_table_ok = 0 (two PRMT tables per step)."""
    mat = matrix_m1().astype(np.int16)
    for b, v in enumerate((0, -1, -2, 1)):
        _sym(mat, 15, b, v)
    return mat.astype(np.int8)


def matrix_asym() -> np.ndarray:
    """M1 made asymmetric: row (read base) and column (candidate base) must not be swapped anywhere."""
    mat = matrix_m1().astype(np.int16)
    mat[0, 1], mat[1, 0] = -4, -8
    mat[2, 3], mat[3, 2] = -1, -9
    for b in range(4):
        mat[b, 14] = -3 - b     # N as a candidate base; the N row stays constant over A/C/G/T
        mat[b, 16] = b - 2
    return mat.astype(np.int8)


MATRICES = {"m1": matrix_m1, "m2": matrix_m2, "asym": matrix_asym}


def packed_ok(mat) -> bool:
    """strk_init (api.cu:284-300): every entry + 2g fits a positive byte."""
    return bool(((mat.astype(np.int16) + 2 * GAP >= 0) & (mat.astype(np.int16) + 2 * GAP <= 127)).all())


def one_table_ok(mat) -> bool:
    return all(len({int(mat[c, b]) for b in range(4)}) == 1 for c in (14, 15, 16))


@pytest.mark.parametrize("name", list(MATRICES))
def test_nonuniform_matrix(sb, oracle, pool, name):
    """Every kernel path under a matrix whose PRMT byte tables hold a distinct value per lane, against an oracle with
    the same matrix: score tables of the width, pairing and gate families, reference tables, whole config-1 / config-3
    batches through count_reads."""
    from strkit_b200 import synth

    mat = MATRICES[name]()
    assert packed_ok(mat) and one_table_ok(mat) == (name != "m2") and (np.array_equal(mat, mat.T) == (name != "asym"))
    o = Oracle(oracle.lib)
    o.matrix = np.ascontiguousarray(mat.reshape(-1), dtype=np.int8)
    assert o.score_candidate("ACGT", "", "", "ACGT", 1, 15) == 3 + 2 + 4 + 1
    fams, lo, hi = read_width_families(5000, classes=(3, 10), widths=(1, 3, 17, 33, 66, 128))
    for part in (paired_families(5001, False), edge_families(5002, False)):
        fams, lo, hi = fams + list(part[0]), lo + list(part[1]), hi + list(part[2])
    for flags in (15, 4):
        check_read(sb, o, pool, fams, lo, hi, flags, matrix=mat, general=flags == 15)
    fams, lo, hi = [], [], []
    for R in (2, 7, 9, 16):
        f, a, b = ref_class_families(R, 5100 + R)
        fams, lo, hi = fams + f[::2], lo + a[::2], hi + b[::2]
    for part in (paired_families(5003, True), edge_families(5004, True)):
        fams, lo, hi = fams + list(part[0]), lo + list(part[1]), hi + list(part[2])
    check_ref(sb, o, pool, fams, lo, hi, matrix=mat)
    params = sb.RepeatCountParams("repalign", 50, 3, 1)
    eng = sb.Engine(matrix=mat)
    for cfg, n_loci in ((1, 60), (3, 30)):
        batch = synth.generate(synth.CONFIGS[cfg], n_loci, seed=60 + cfg).to_host()
        got = eng.count_reads(batch, params)
        want, _ = o.count_loci(batch.arena, batch.seq_off, batch.lens, batch.est_cn, batch.read_begin, batch.motif_off,
                               batch.motif_len, n_threads=16)
        assert np.array_equal(got, want), (cfg, np.flatnonzero((got != want).any(axis=1))[:10])
        assert eng.stats()["reads_packed_kernel"] > 0
    eng.close()


# ------------------------------------------------------------------------------------------------ 6. work queue
def tiled_batch(base: ReadBatch, idx: np.ndarray) -> ReadBatch:
    """Families base[idx] (one read per locus) sharing the base arena."""
    n = idx.shape[0]
    return ReadBatch(arena=base.arena, seq_off=base.seq_off[idx].copy(), lens=base.lens[idx].copy(),
                     est_cn=base.est_cn[idx].copy(), read_begin=np.arange(n + 1, dtype=np.int64),
                     motif_off=base.motif_off[idx].copy(), motif_len=base.motif_len[idx].copy())


@pytest.mark.parametrize("n", [131072, 131073])
def test_work_queue_large_lists(sb, oracle, pool, n):
    """Class lists several times longer than the resident warps (16 and 32 lanes): the queue is popped one read ahead,
    then after the read near its end; ineligible reads spread through the lists fall back while the next item is
    held.  131 072 families fan the classes out on side streams with disjoint scratch slices, one more launches them
    back to back.  Every entry against the general kernel, a seeded sample against the oracle."""
    rng = np.random.default_rng(6000)
    fams = []
    for i in range(4096):
        R = (4, 4, 4, 10, 10, 13, 2)[i % 7]
        f = class_family(rng, R, i % 5)
        if i % 97 == 5:   # an IUPAC code inside the read
            f = (f[0], f[1][:3] + "Y" + f[1][4:], f[2], f[3]) if len(f[1]) > 4 else f
        fams.append(f)
    base = families_to_batch(fams)
    wins = [window(f, 1 + i % 4) for i, f in enumerate(fams)]
    idx = rng.integers(0, len(fams), size=n)
    batch = tiled_batch(base, idx)
    lo = np.array([wins[i][0] for i in idx], dtype=np.int32)
    hi = np.array([wins[i][1] for i in idx], dtype=np.int32)
    sub_fams = [fams[i] for i in idx]
    counts = np.bincount([pk_class(len(fams[i][2]), len(fams[i][1]), len(fams[i][3]), len(fams[i][0])) for i in idx],
                         minlength=17)
    resident = 148 * (2048 // 128) * 4   # warps of 4-warp CTAs a B200 can hold at once, whatever the occupancy
    assert counts[4] > 2 * 2 * resident and counts[10] > 2 * resident
    eng = sb.Engine()
    got, off = eng.score_tables(batch, lo, hi)
    st = eng.stats()
    kept = predict_packed(sub_fams, lo, hi, ref=False)
    assert (st["reads_packed_kernel"], st["reads_general_kernel"]) == (kept, n - kept) and kept < n - 300
    want, _ = eng.score_tables(batch, lo, hi, kernel=sb.KERNEL_GENERAL)
    assert np.array_equal(got, want), np.flatnonzero(got != want)[:10]
    sample = np.sort(rng.choice(n, size=400, replace=False))
    s_fams = [sub_fams[i] for i in sample]
    w = oracle_read_tables(oracle, pool, s_fams, lo[sample], hi[sample], 15)
    g = np.concatenate([got[int(off[i]): int(off[i]) + int(hi[i] - lo[i]) + 1] for i in sample])
    assert np.array_equal(g, w)
    eng.close()


# ------------------------------------------------------------------------------------------------ 7. widening pass
@pytest.mark.parametrize("long_motif", [False, True])
def test_widening_pass_merged_classes(sb, oracle, long_motif):
    """count_reads whose bad estimates send loci of several classes of each lane group to a second pass: a small
    pass runs them merged in the largest class of their group (widening_pass in api.cu), hundreds of pad rows above the
    short reads.  With a 64-base motif in the 16-lane group the merged tables pass the shared-memory limit and that
    segment runs on the general kernel instead (launch_pass).  Global alignment (end flags 0): every copy
    beyond the tract costs, so each search walks from its estimate to the tract's count and leaves the first window."""
    rng = np.random.default_rng(7000 + long_motif)
    loci, classes = [], set()
    for j, R in enumerate((2, 3, 5, 8, 9, 11, 14, 16) * 2):
        off = R in (2, 5, 8, 9, 14, 16)          # these loci's estimates are far off: they go to a second pass
        m = 64 if (long_motif and j == 0) else int(rng.integers(1, min(6, 128 // R) + 1))
        motif = rand_seq(rng, m)
        n1 = int(rng.integers(32 * (R - 1), 32 * R))
        f_hi = min(40, n1 // 2 - 2)
        fl, fr = (10, 10) if m == 64 else (int(rng.integers(5, f_hi)), int(rng.integers(5, f_hi)))
        trs = [periodic(rng, motif, n1 - fl - fr) for _ in range(3)]
        est = [round(len(t) / m) + (int(rng.integers(12, 20)) if off else 0) for t in trs]
        loci.append(LocusReads(motif, est, trs, [rand_seq(rng, fl) for _ in trs], [rand_seq(rng, fr) for _ in trs]))
        classes.add(pk_class(fl, n1 - fl - fr, fr, m))
    assert classes == {2, 3, 5, 8, 9, 11, 14, 16}
    batch = pack_loci(loci)
    params = sb.RepeatCountParams("repalign", 50, 3, 1)
    eng = sb.Engine(end_flags=0)
    got = eng.count_reads(batch, params)
    st = eng.stats()
    want, _ = oracle.count_loci(batch.arena, batch.seq_off, batch.lens, batch.est_cn, batch.read_begin,
                                batch.motif_off, batch.motif_len, flags=0, n_threads=16)
    assert np.array_equal(got, want), np.flatnonzero((got != want).any(axis=1))[:10]
    assert st["widening_passes"] >= 1 and st["reads_packed_kernel"] > 0
    assert np.array_equal(eng.count_reads(batch, params, kernel=sb.KERNEL_GENERAL), want)
    eng.close()
