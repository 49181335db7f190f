"""Batch planning: the host planner (batches of at most 512 reads) and the device planner (plan.cuh, larger batches)
apply one set of read, locus and estimate rules.  Every error kind gives the same code and text on both; one set of
loci gets the same classes, scratch and results from both; the direct entry points word the same rules their own way."""
import numpy as np
import pytest

from tests.helpers import families_to_batch, rand_seq

pytestmark = pytest.mark.gpu

SMALL_BATCH = 512  # api.cu STRK_SMALL_BATCH: larger batches are planned on the device
F = 3              # index of the faulty read / locus (one read per locus: the same index)
BASE = ("CAG", "CAG" * 6, "ACGTTGCA", "TGCAACGT")


@pytest.fixture(scope="module")
def sb():
    import strkit_b200

    assert strkit_b200.device_count() > 0, "no CUDA device: these tests must run on the GPU box"
    return strkit_b200


@pytest.fixture(scope="module")
def eng(sb):
    e = sb.Engine()
    yield e
    e.close()


def _raises(fn, message):
    from strkit_b200._native import StrkError

    with pytest.raises(StrkError) as exc:
        fn()
    assert exc.value.code == 1 and str(exc.value) == f"strkit_b200 native error 1: {message}"


def _set(name, index, value):
    def f(b):
        getattr(b, name)[index] = value
    return f


def _both(*fs):
    def f(b):
        for g in fs:
            g(b)
    return f


# (case, family at F or None, fault, message or None = the batch is valid)
PLAN_CASES = [
    ("neg_len", None, _set("lens", (F, 1), -1), f"batch: read {F} has a negative length"),
    ("empty", None, _set("lens", F, (0, 0, 0)), f"batch: read {F} is empty (fl + tr + fr has no bases)"),
    ("too_long", None, _set("lens", F, (0, (1 << 24) + 1, 0)), f"batch: read {F} is too long"),
    ("longest", None, _set("lens", F, (0, 1 << 24, 0)), f"batch: read {F} runs past the end of the arena"),
    ("past_arena", None, lambda b: _set("seq_off", F, np.uint64(b.arena.nbytes - 5))(b),
     f"batch: read {F} runs past the end of the arena"),
    ("seq_off_wraps", None, _set("seq_off", F, np.uint64(2 ** 64 - 4)), f"batch: read {F} runs past the end of the arena"),
    ("est_negative", None, _set("est_cn", F, -1), f"batch: read {F} has an out-of-range est_cn"),
    ("est_zero", None, _set("est_cn", F, 0), None),
    ("est_above_2^22", ("C", "C" * 10, "AGTA", "GTAG"), _set("est_cn", F, (1 << 22) + 1),
     f"batch: read {F} has an out-of-range est_cn"),
    ("m_est_at_2^24", ("CAGT", "CAGT" * 4, "AGTA", "GTAG"), _set("est_cn", F, 1 << 22), None),
    ("m_est_above_2^24", ("CAGTA", "CAGTA" * 4, "AGTA", "GTAG"), _set("est_cn", F, 1 << 22),
     f"batch: read {F} has an out-of-range est_cn"),
    ("motif_empty", None, _set("motif_len", F, 0), f"batch: locus {F} has an empty motif"),
    ("motif_past_arena", None, lambda b: _set("motif_off", F, np.uint64(b.arena.nbytes - 1))(b),
     f"batch: locus {F} has a motif that runs past the end of the arena"),
    ("motif_off_wraps", None, _set("motif_off", F, np.uint64(2 ** 64 - 2)),
     f"batch: locus {F} has a motif that runs past the end of the arena"),
    ("read_begin_falls", None, _set("read_begin", F + 1, F - 1), f"batch: locus {F} has a non-monotone read_begin"),
    ("read_begin_past_reads", None, lambda b: _set("read_begin", F + 1, b.n_reads + 5)(b),
     f"batch: locus {F} has a non-monotone read_begin"),
    ("locus_after_read", None, _both(_set("lens", (1, 1), -1), _set("motif_len", F + 2, 0)),
     f"batch: locus {F + 2} has an empty motif"),
]


@pytest.mark.parametrize("n_loci", [8, 600], ids=["host_planner", "device_planner"])
@pytest.mark.parametrize("case,special,fault,message", PLAN_CASES, ids=[c[0] for c in PLAN_CASES])
def test_plan_errors_both_planners(sb, eng, n_loci, case, special, fault, message):
    fams = [BASE] * n_loci
    if special:
        fams[F] = special
    b = families_to_batch(fams)
    fault(b)
    assert (b.n_reads <= SMALL_BATCH) == (n_loci == 8)
    if message is None:
        eng.upload(b).free()
    else:
        _raises(lambda: eng.upload(b), message)


def _plan_mix(rng):
    """512 loci of one read each: packed classes of 16 and 32 lanes, general-kernel reads, IUPAC reads, long reads.
    Exact tracts and est = the tract's copies keep every search inside its first window."""
    fams, est = [], []

    def add(motif, k, fl, fr, iupac=False):
        tr = motif * k
        if iupac:
            tr = tr[: len(tr) // 2] + "R" + tr[len(tr) // 2 + 1:]
        fams.append((motif, tr, rand_seq(rng, fl), rand_seq(rng, fr)))
        est.append(k)

    def motif(m):
        return rand_seq(rng, m)

    for i in range(512):
        kind = i % 8
        if kind in (0, 1):    # 16 lanes: db <= 256
            m = int(rng.integers(1, 7))
            add(motif(m), int(rng.integers(3, 120 // m + 4)), int(rng.integers(5, 61)), int(rng.integers(5, 61)))
        elif kind in (2, 3):  # 32 lanes: db of 257..512
            m = int(rng.integers(1, 9))
            add(motif(m), int(rng.integers(130 // m + 1, 340 // m + 1)), 70, 70)
        elif kind == 4:       # general kernel: an empty flank, a flank past 160, m * R > 128
            j = i // 8 % 3
            if j == 0:
                add(motif(3), int(rng.integers(5, 40)), 0, 40)
            elif j == 1:
                add(motif(4), int(rng.integers(5, 40)), 200, 50)
            else:
                add(motif(10), int(rng.integers(25, 37)), 70, 70)
        elif kind == 5:       # IUPAC code in the tract: the packed kernel hands the read back to the general kernel
            # (32 lanes: one read per warp, so no other read goes back with it, whatever order a planner lists them in)
            m = int(rng.integers(2, 6))
            add(motif(m), int(rng.integers(130 // m + 1, 340 // m + 1)), 70, 70, iupac=True)
        elif kind == 6:       # more than one 512-row strip
            m = int(rng.integers(2, 7))
            add(motif(m), int(rng.integers(600 // m, 1500 // m)), 70, 70)
        else:
            m = int(rng.integers(2, 6))
            add(motif(m), int(rng.integers(5, 60)), 50, 50)
    return fams, est


def test_same_plan_both_planners(sb, oracle):
    rng = np.random.default_rng(77)
    fams, est = _plan_mix(rng)
    params = sb.RepeatCountParams("repalign", 50, 3, 1)
    runs = []
    for extra in ([], [("CAGT", "CAGT" * 12, "ACGTTGCAAG", "TGCAACGTTC")]):
        b = families_to_batch(fams + extra, est=est + [12] * len(extra))
        e = sb.Engine()  # (a fresh context: the first-window policy is carried in the context's reused batch)
        got = e.count_reads(b, params)
        st = e.stats()
        e.close()
        want, _ = oracle.count_loci(b.arena, b.seq_off, b.lens, b.est_cn, b.read_begin, b.motif_off, b.motif_len,
                                    n_threads=8)
        assert np.array_equal(got, want), np.flatnonzero((got != want).any(axis=1))[:10]
        assert st["widening_passes"] == 0
        runs.append((b.n_reads, got, st))
    (n_host, got_host, st_host), (n_dev, got_dev, st_dev) = runs
    assert n_host == SMALL_BATCH and n_dev == SMALL_BATCH + 1
    assert np.array_equal(got_dev[:n_host], got_host)
    assert st_host["reads_general_kernel"] > 0 and st_host["reads_packed_kernel"] > 0
    assert st_dev["reads_packed_kernel"] == st_host["reads_packed_kernel"] + 1
    assert st_dev["reads_general_kernel"] == st_host["reads_general_kernel"]


TABLE_CASES = [
    ("too_long", _set("lens", 1, (0, (1 << 24) + 1, 0)), "{who}: read 1 is too long (16777217)"),
    ("seq_off_wraps", _set("seq_off", 1, np.uint64(2 ** 64 - 4)), "{who}: read 1 runs past the end of the arena"),
    ("motif_empty", _set("motif_len", 1, 0), "{who}: motif 1 is empty"),
    ("motif_past_arena", lambda b: _set("motif_off", 1, np.uint64(b.arena.nbytes - 1))(b),
     "{who}: motif 1 runs past the end of the arena"),
    ("read_before_motif", _both(_set("lens", (2, 0), -1), _set("motif_len", 0, 0)), "{who}: read 2 has a negative length"),
]


@pytest.mark.parametrize("case,fault,message", TABLE_CASES, ids=[c[0] for c in TABLE_CASES])
def test_table_entry_point_messages(sb, eng, case, fault, message):
    b = families_to_batch([BASE] * 4)
    fault(b)
    n_lo, n_hi = np.full(4, 4), np.full(4, 8)
    _raises(lambda: eng.score_tables(b, n_lo, n_hi), message.format(who="strk_score_tables"))
    _raises(lambda: eng.ref_boundary_tables(b, n_lo, n_hi), message.format(who="strk_ref_boundary_tables"))


REF_CASES = [
    ("empty", None, _set("lens", 1, (0, 0, 0)), "strk_ref_counts: read 1 is empty (fl + tr + fr has no bases)"),
    ("past_arena", None, lambda b: _set("seq_off", 1, np.uint64(b.arena.nbytes - 5))(b),
     "strk_ref_counts: read 1 runs past the end of the arena"),
    ("motif_off_wraps", None, _set("motif_off", 1, np.uint64(2 ** 64 - 2)),
     "strk_ref_counts: motif 1 runs past the end of the arena"),
    ("start_negative", None, lambda b: None, "strk_ref_counts: bad start count / search parameters for locus 1"),
    ("m_start_above_2^24", ("CAGTA", "CAGTA" * 4, "AGTA", "GTAG"), lambda b: None,
     "strk_ref_counts: bad start count / search parameters for locus 1"),
    ("read_before_motif", None, _both(_set("lens", (2, 2), -1), _set("motif_len", 0, 0)),
     "strk_ref_counts: read 2 has a negative length"),
]


@pytest.mark.parametrize("case,special,fault,message", REF_CASES, ids=[c[0] for c in REF_CASES])
def test_ref_counts_messages(sb, eng, case, special, fault, message):
    fams = [BASE] * 4
    if special:
        fams[1] = special
    b = families_to_batch(fams)
    fault(b)
    start = np.full(4, 6, dtype=np.int32)
    if case == "start_negative":
        start[1] = -1
    elif case == "m_start_above_2^24":
        start[1] = 1 << 22
    rc = np.tile(np.array([50, 3, 1], dtype=np.int32), (4, 1))
    _raises(lambda: eng.ref_counts(b, start, np.full(4, 18, dtype=np.int32), rc, 1), message)
