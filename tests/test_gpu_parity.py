"""Parity tests proper: the CUDA path (through the C ABI) against the CPU oracle, bit-exact.
Run on the GPU box with `pytest -m gpu`."""
import numpy as np
import pytest

from tests.helpers import families_to_batch, mutate, oracle_tables, random_families

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sb():
    import strkit_b200

    assert strkit_b200.device_count() > 0, "no CUDA device: these tests must run on the GPU box"
    return strkit_b200


@pytest.mark.parametrize("kernel", ["auto", "general"])
@pytest.mark.parametrize("flags", list(range(16)))
def test_score_tables_all_modes_small(sb, oracle, flags, kernel):
    rng = np.random.default_rng(100 + flags)
    fams = random_families(rng, 120)
    n_lo, n_hi = [], []
    for motif, tr, fl, fr in fams:
        e = round(len(tr) / len(motif))
        lo = max(0, e - int(rng.integers(0, 5)))
        if lo == 0 and len(fl) + len(fr) == 0:
            lo = 1  # an empty candidate has no alignment
        n_lo.append(lo)
        n_hi.append(lo + int(rng.integers(0, 9)))
    eng = sb.Engine(end_flags=flags)
    got, _ = eng.score_tables(families_to_batch(fams), np.array(n_lo), np.array(n_hi),
                              kernel=sb.KERNEL_GENERAL if kernel == "general" else sb.KERNEL_AUTO)
    want = oracle_tables(oracle, fams, n_lo, n_hi, flags)
    assert np.array_equal(got, want), np.flatnonzero(got != want)[:10]
    st = eng.stats()
    if kernel == "auto":  # most of these families are eligible for the packed u16x2 kernel
        assert st["reads_packed_kernel"] > 40 and st["reads_general_kernel"] > 0
    else:
        assert st["reads_packed_kernel"] == 0
    eng.close()


@pytest.mark.parametrize("flags", [0, 2, 5, 10, 15])
def test_score_tables_packed_kernel_realistic_lengths(sb, oracle, flags):
    """Read-sized families (db 100-510 bases, every packed R), wide windows, X / N wildcards, lower case."""
    rng = np.random.default_rng(200 + flags)
    fams, n_lo, n_hi = [], [], []
    for i in range(64):
        m = int(rng.integers(1, 9))
        motif = "".join(rng.choice(list("ACGT"), size=m))
        k = int(rng.integers(1, max(2, 370 // m)))
        tr = mutate(rng, motif * k, 0.03, 0.02, 0.02)[:370]
        fl = "".join(rng.choice(list("ACGT"), size=int(rng.integers(1, 71))))
        fr = "".join(rng.choice(list("ACGT"), size=int(rng.integers(1, 71))))
        if i % 3 == 0:
            tr = "".join("X" if rng.random() < 0.03 else ("N" if rng.random() < 0.01 else ch) for ch in tr)
            fl = "".join("X" if rng.random() < 0.03 else ch for ch in fl)
            fr = "".join("N" if rng.random() < 0.03 else ch for ch in fr)
        if i % 5 == 0:
            tr, fl = tr.lower(), fl.lower()
        e = round(len(tr) / m)
        lo = max(0, e - int(rng.integers(0, 12)))
        fams.append((motif, tr or "A", fl, fr))
        n_lo.append(lo)
        n_hi.append(lo + int(rng.integers(0, 24)))
    eng = sb.Engine(end_flags=flags)
    got, _ = eng.score_tables(families_to_batch(fams), np.array(n_lo), np.array(n_hi))
    want = oracle_tables(oracle, fams, n_lo, n_hi, flags)
    assert np.array_equal(got, want), np.flatnonzero(got != want)[:10]
    assert eng.stats()["reads_packed_kernel"] == len(fams)
    eng.close()


def test_score_tables_known_answers(sb):
    """SURVEY 8c: exact tract => score(k) = 2L, score(k+1) = 2L - 5m (any mode)."""
    rng = np.random.default_rng(5)
    eng = sb.Engine()
    fams, ks = [], []
    for _ in range(32):
        m = int(rng.integers(2, 7))
        while True:
            motif = "".join(rng.choice(list("ACGT"), size=m))
            if all(motif != motif[p:] + motif[:p] for p in range(1, m)):
                break
        k = int(rng.integers(8, 60))
        while True:
            fl = "".join(rng.choice(list("ACGT"), size=70))
            fr = "".join(rng.choice(list("ACGT"), size=70))
            if fl[-m:] != motif and fr[:m] != motif:
                break
        fams.append((motif, motif * k, fl, fr))
        ks.append(k)
    ks = np.array(ks)
    got, off = eng.score_tables(families_to_batch(fams), ks, ks + 1)
    for i, (motif, tr, fl, fr) in enumerate(fams):
        L = 140 + len(tr)
        assert got[int(off[i])] == 2 * L and got[int(off[i]) + 1] == 2 * L - 5 * len(motif)


def test_get_repeat_count_golden(sb, golden):
    """The drop-in per-call API against the committed vectors (reference dispatcher + restated search)."""
    for c in golden["read_restated"]:
        params = sb.RepeatCountParams("repalign", c["max_iters"], c["local_search_range"], c["step_size"])
        (n, s), n_exp, delta = sb.get_repeat_count(c["start_count"], c["tr_seq"], c["flank_left_seq"],
                                                   c["flank_right_seq"], c["motif"], params)
        assert [n, s, n_exp, delta] == c["expect"], c


def test_batch_config1_bit_exact(sb, oracle):
    from strkit_b200 import synth

    batch = synth.generate(synth.CONFIGS[1], 300, seed=11).to_host()
    params = sb.RepeatCountParams("repalign", 50, 3, 1)
    eng = sb.Engine()
    got = eng.count_reads(batch, params)
    want, cells = oracle.count_loci(batch.arena, batch.seq_off, batch.lens, batch.est_cn, batch.read_begin,
                                    batch.motif_off, batch.motif_len, n_threads=8)
    assert np.array_equal(got, want), np.flatnonzero((got != want).any(axis=1))[:10]
    st = eng.stats()
    assert st["reference_cells"] == cells  # the replay scored exactly the sizes the reference scores
    assert 0 < st["executed_cells"] < cells
    # HiFi reads all take the packed u16x2 kernel (identical reads of a locus share one table when STRK_DEDUPE is on)
    assert st["reads_general_kernel"] == 0 and 0.5 * batch.n_reads < st["reads_packed_kernel"] <= batch.n_reads
    got_general = eng.count_reads(batch, params, kernel=sb.KERNEL_GENERAL)
    assert np.array_equal(got_general, want) and eng.stats()["reads_packed_kernel"] == 0


def test_count_reads_stream_matches_blocking_calls_and_oracle(sb, oracle):
    """Streamed locus blocks (two contexts, two host threads, copies overlapped with kernels): same results,
    in block order, as one blocking call per block; blocks of different sizes, an empty block in between."""
    from strkit_b200 import synth

    params = sb.RepeatCountParams("repalign", 50, 3, 1)
    blocks = [synth.generate(synth.CONFIGS[c], n, seed=40 + i).to_host()
              for i, (c, n) in enumerate([(1, 120), (3, 40), (1, 1), (2, 200), (1, 64), (3, 10), (2, 33)])]
    blocks.insert(3, blocks[0].slice_loci(0, 0))  # no loci, no reads
    eng = sb.Engine()
    got = list(eng.count_reads_stream(blocks, params))
    assert len(got) == len(blocks)
    for b, g in zip(blocks, got):
        assert g.shape == (b.n_reads, 4)
        if b.n_reads == 0:
            continue
        assert np.array_equal(g, eng.count_reads(b, params))
        want, _ = oracle.count_loci(b.arena, b.seq_off, b.lens, b.est_cn, b.read_begin, b.motif_off, b.motif_len,
                                    n_threads=8)
        assert np.array_equal(g, want)
    # caller-provided output buffers are filled in place
    outs = [np.full((b.n_reads, 4), -7, dtype=np.int32) for b in blocks]
    for b, o, g in zip(blocks, eng.count_reads_stream(blocks, params, outs=outs), got):
        assert np.array_equal(o, g)
    assert all(np.array_equal(o, g) for o, g in zip(outs, got))
    eng.close()


def test_small_pinned_batch_owns_nothing_after_upload_and_runs_on_a_foreign_stream(sb, oracle):
    """include/strkit_b200.h: the library keeps no host pointer after a call returns.  A block of <= 512 reads (planned
    on the host, copies queued asynchronously from PINNED arrays) is uploaded, every host array is overwritten at once,
    and the batch runs on a stream the library does not own: results must be those of the arrays as uploaded."""
    import torch

    from strkit_b200 import synth
    from strkit_b200.batcher import ReadBatch

    params = sb.RepeatCountParams("repalign", 50, 3, 1)
    eng = sb.Engine()
    foreign = torch.cuda.Stream()
    for seed, n_loci, nibble in ((3, 12, False), (4, 16, True), (5, 1, False)):
        b = synth.generate(synth.CONFIGS[1], n_loci, seed=900 + seed).to_host(pin=True, nibble=nibble)
        assert 0 < b.n_reads <= 512
        keep = ReadBatch(arena=b.arena.copy(), seq_off=b.seq_off.copy(), lens=b.lens.copy(), est_cn=b.est_cn.copy(),
                         read_begin=b.read_begin.copy(), motif_off=b.motif_off.copy(), motif_len=b.motif_len.copy(),
                         arena_format=b.arena_format)
        db = eng.upload(b)
        b.arena[:] = 0x58 if not nibble else 0xFF  # the caller reuses its buffers straight away
        b.seq_off[:] = 0
        b.lens[:] = 1
        b.est_cn[:] = 0
        b.motif_off[:] = 0
        b.motif_len[:] = 1
        with torch.cuda.stream(foreign):
            eng.run(db, params, stream=foreign.cuda_stream)
        foreign.synchronize()
        got = eng.download(db)
        db.free()
        a = keep.to_ascii() if nibble else keep
        want, _ = oracle.count_loci(a.arena, a.seq_off, a.lens, a.est_cn, a.read_begin, a.motif_off, a.motif_len, n_threads=4)
        assert np.array_equal(got, want)
    eng.close()


def test_batch_noisy_ont_and_bad_estimates_force_widening(sb, oracle):
    """Config-3-like reads with start estimates far off: the search leaves the first table window and
    the widening passes must still reproduce the reference trajectory exactly."""
    from strkit_b200 import synth

    batch = synth.generate(synth.CONFIGS[3], 60, seed=12).to_host()
    rng = np.random.default_rng(3)
    est = batch.est_cn.copy()
    bad = rng.random(est.shape[0]) < 0.2
    est[bad] = np.maximum(0, est[bad] + rng.integers(-30, 60, int(bad.sum())))
    batch.est_cn = est.astype(np.int32)
    params = sb.RepeatCountParams("repalign", 50, 3, 1)
    eng = sb.Engine()
    got = eng.count_reads(batch, params)
    want, _ = oracle.count_loci(batch.arena, batch.seq_off, batch.lens, batch.est_cn, batch.read_begin,
                                batch.motif_off, batch.motif_len, n_threads=8)
    assert np.array_equal(got, want), np.flatnonzero((got != want).any(axis=1))[:10]
    assert eng.stats()["widening_passes"] >= 1


def test_first_window_policy_changes_passes_not_results(sb, oracle, monkeypatch):
    """Noisy reads switch the blocks that follow to the wider first window for short motifs (strk_read_wd) and the
    small second passes run merged in the largest class of their lane group: same rows as the oracle whichever
    window a block was scored with -- policy learnt (2nd call), forced on, forced off, 8x first widening."""
    from strkit_b200 import synth

    batch = synth.generate(synth.CONFIGS[3], 512, seed=77).to_host()
    params = sb.RepeatCountParams("repalign", 50, 3, 1)
    want, _ = oracle.count_loci(batch.arena, batch.seq_off, batch.lens, batch.est_cn, batch.read_begin,
                                batch.motif_off, batch.motif_len, n_threads=8)
    eng = sb.Engine()
    got = eng.count_reads(batch, params)
    assert np.array_equal(got, want)
    assert eng.stats()["widening_passes"] >= 1          # +-6 copies: some 2-mer loci leave the window
    first_pass_reads = eng.stats()["reads_packed_kernel"] + eng.stats()["reads_general_kernel"]
    got = eng.count_reads(batch, params)                # same batch object: the policy is on now
    assert np.array_equal(got, want)
    assert eng.stats()["reads_packed_kernel"] + eng.stats()["reads_general_kernel"] < first_pass_reads
    for env in ({"STRK_WIDE_SHORT": "1"}, {"STRK_WIDE_SHORT": "0"}, {"STRK_WIDE_SHORT": "0", "STRK_WIDEN1": "8"}):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        assert np.array_equal(eng.count_reads(batch, params), want), env
    eng.close()


def test_identical_reads_share_tables(sb, oracle, monkeypatch):
    """Identical reads of a locus (same flanks, tract, estimate) run the DP once; the replay still runs
    per read.  HiFi-like blocks (a third of the reads are duplicates), the same sequence with two different estimates,
    bad estimates that force second passes, and an ONT-like block without duplicates: rows equal the oracle's."""
    from strkit_b200 import synth

    monkeypatch.delenv("STRK_DEDUPE", raising=False)
    params = sb.RepeatCountParams("repalign", 50, 3, 1)
    eng = sb.Engine()
    for cfg, n_loci, tweak in ((2, 700, None), (2, 700, "est"), (2, 700, "bad"), (3, 300, None)):
        batch = synth.generate(synth.CONFIGS[cfg], n_loci, seed=40 + cfg).to_host()
        rng = np.random.default_rng(8)
        est = batch.est_cn.copy()
        if tweak == "est":   # same bytes, different start estimate: must not share a table row's window
            est[rng.random(est.shape[0]) < 0.3] += 1
        if tweak == "bad":
            bad = rng.random(est.shape[0]) < 0.05
            est[bad] = np.maximum(0, est[bad] + rng.integers(-30, 60, int(bad.sum())))
        batch.est_cn = est.astype(np.int32)
        got = eng.count_reads(batch, params)
        want, cells = oracle.count_loci(batch.arena, batch.seq_off, batch.lens, batch.est_cn, batch.read_begin,
                                        batch.motif_off, batch.motif_len, n_threads=8)
        assert np.array_equal(got, want), (cfg, tweak, np.flatnonzero((got != want).any(axis=1))[:10])
        st = eng.stats()
        computed = st["reads_packed_kernel"] + st["reads_general_kernel"]
        if cfg == 2 and tweak is None:
            assert st["reference_cells"] == cells
            assert 0.5 * batch.n_reads < computed < 0.8 * batch.n_reads   # ~33 % of the reads share a table
        if cfg == 3:
            assert computed >= batch.n_reads                              # nothing to share
        monkeypatch.setenv("STRK_DEDUPE", "0")                            # measurement switch: every read its own table
        assert np.array_equal(eng.count_reads(batch, params), want)
        st = eng.stats()
        assert st["reads_packed_kernel"] + st["reads_general_kernel"] >= batch.n_reads
        monkeypatch.delenv("STRK_DEDUPE")
    eng.close()


@pytest.mark.parametrize("params", [(7, 3, 1), (50, 3, 2), (50, 1, 4), (200, 3, 3), (0, 3, 1)])
def test_batch_search_parameters(sb, oracle, params):
    from strkit_b200 import synth
    from strkit_b200._native import StrkError

    batch = synth.generate(synth.CONFIGS[1], 40, seed=13).to_host()
    p = sb.RepeatCountParams("repalign", *params)
    eng = sb.Engine()
    if params[0] == 0:  # nothing scored: the reference raises ValueError (max() of an empty dict)
        with pytest.raises(StrkError):
            eng.count_reads(batch, p)
        return
    got = eng.count_reads(batch, p)
    want, _ = oracle.count_loci(batch.arena, batch.seq_off, batch.lens, batch.est_cn, batch.read_begin,
                                batch.motif_off, batch.motif_len, max_iters=params[0], local_search_range=params[1],
                                step_size=params[2], n_threads=8)
    assert np.array_equal(got, want)


# (50, 3, 1): first windows of 13 sizes, replayed by replay_reads_small_kernel; (50, 8, 3): 27 sizes, replay_reads_kernel
@pytest.mark.parametrize("tie,search", [pytest.param(t, s, id=f"{t}{sfx}") for s, sfx in [((50, 3, 1), ""), ((50, 8, 3), "-w27")]
                                        for t in [1, 2, 3, 4, 8, 7]])
def test_tie_break_switches(sb, oracle, tie, search):
    rng = np.random.default_rng(9)
    # homopolymer-ish tracts with wildcards produce many equal scores
    fams = [("A", "A" * int(rng.integers(3, 20)) + "X" * int(rng.integers(0, 4)), "", "ACGTT") for _ in range(40)]
    batch = families_to_batch(fams, est=[int(rng.integers(0, 25)) for _ in fams])
    eng = sb.Engine(tie_flags=tie)
    got = eng.count_reads(batch, sb.RepeatCountParams("repalign", *search))
    want, _ = oracle.count_loci(batch.arena, batch.seq_off, batch.lens, batch.est_cn, batch.read_begin,
                                batch.motif_off, batch.motif_len, max_iters=search[0], local_search_range=search[1],
                                step_size=search[2], tie_flags=tie)
    assert np.array_equal(got, want)


@pytest.mark.parametrize("policy", [4, 8, 5, 10])
@pytest.mark.parametrize("cfg,search", [(2, (50, 3, 1)), (3, (50, 3, 1)), (3, (30, 7, 2)), (2, (12, 2, 3))])
def test_search_policy_switches(sb, oracle, policy, cfg, search):
    """STRK_SEARCH_NARROW_FIRST / _HALVE (with and without a tie switch): the range-narrowing hypotheses about the Rust
    body of get_repeat_count (repeat_count_params.py:13) are switches of the replay and of the oracle, not assumptions;
    each one is bit-exact against the oracle run with the same flags, and it changes n_explored on most reads."""
    from strkit_b200 import synth

    batch = synth.generate(synth.CONFIGS[cfg], 300, seed=77 + cfg).to_host()
    rng = np.random.default_rng(policy)
    est = batch.est_cn.copy()
    off = rng.random(est.shape[0]) < 0.1   # some bad starts: long climbs, iteration budget, second passes
    est[off] = np.maximum(0, est[off] + rng.integers(-12, 13, int(off.sum())))
    batch.est_cn = est.astype(np.int32)
    params = sb.RepeatCountParams("repalign", *search)
    eng = sb.Engine(tie_flags=policy)
    got = eng.count_reads(batch, params)
    want, _ = oracle.count_loci(batch.arena, batch.seq_off, batch.lens, batch.est_cn, batch.read_begin, batch.motif_off,
                                batch.motif_len, max_iters=search[0], local_search_range=search[1], step_size=search[2],
                                tie_flags=policy, n_threads=8)
    assert np.array_equal(got, want), np.flatnonzero((got != want).any(axis=1))[:10]
    base, _ = oracle.count_loci(batch.arena, batch.seq_off, batch.lens, batch.est_cn, batch.read_begin, batch.motif_off,
                                batch.motif_len, max_iters=search[0], local_search_range=search[1], step_size=search[2],
                                tie_flags=policy & 3, n_threads=8)
    assert (want[:, 2] <= base[:, 2]).mean() > 0.95 and (want[:, 2] < base[:, 2]).mean() > 0.5
    eng.close()


def test_long_expansions_multi_pass(sb, oracle):
    """Config-4-like: tracts longer than one 512-row strip, IUPAC motifs, int32 range."""
    from strkit_b200 import synth

    batch, _ = synth.generate_expansions(n_loci=6, reads_per_locus=4, max_tract=1800, big_lo=150, big_hi=400)
    eng = sb.Engine()
    params = sb.RepeatCountParams("repalign", 50, 3, 1)
    got = eng.count_reads(batch, params)
    want, _ = oracle.count_loci(batch.arena, batch.seq_off, batch.lens, batch.est_cn, batch.read_begin,
                                batch.motif_off, batch.motif_len, n_threads=8)
    assert np.array_equal(got, want), (got[:8], want[:8])


@pytest.mark.parametrize("flags", [0, 6, 9, 15])
def test_general_kernel_many_strips(sb, oracle, flags):
    """Reads of 6 to 13 strips of 512 rows: the strips run as a pipeline over the 4 warps of a CTA and the ring of
    boundary rows (5 slots) is reused -- DUMP / COMBINE sweeps here, ARGMAX in the reference-boundary test below."""
    rng = np.random.default_rng(300 + flags)
    fams, n_lo, n_hi = [], [], []
    for k, motif in ((520, "CAGGT"), (1400, "AAG"), (1290, "GGCCT"), (2200, "CTG"), (6100, "A")):
        tr = mutate(rng, motif * k, 0.01, 0.005, 0.005)
        if k == 1400:
            tr = "".join("X" if rng.random() < 0.01 else ("R" if rng.random() < 0.002 else ch) for ch in tr)  # look-up path
        fl = "".join(rng.choice(list("ACGT"), size=70))
        fr = "".join(rng.choice(list("ACGT"), size=int(rng.integers(1, 71))))
        fams.append((motif, tr, fl, fr))
        e = round(len(tr) / len(motif))
        n_lo.append(e - 1)
        n_hi.append(e + 1)
    eng = sb.Engine(end_flags=flags)
    got, _ = eng.score_tables(families_to_batch(fams), np.array(n_lo), np.array(n_hi), kernel=sb.KERNEL_GENERAL)
    want = oracle_tables(oracle, fams, n_lo, n_hi, flags)
    assert np.array_equal(got, want), np.flatnonzero(got != want)[:10]
    eng.close()


def test_ref_boundary_tables_many_strips(sb, oracle):
    """score_ref_boundaries on reference windows of 7 and 10 strips (ARGMAX sweeps of the general kernel)."""
    rng = np.random.default_rng(77)
    fams, ns = [], []
    for k, motif in ((1100, "CAG"), (980, "GGCCT")):
        tr = mutate(rng, motif * k, 0.004, 0.002, 0.002)
        fams.append((motif, tr, "".join(rng.choice(list("ACGT"), size=70)), "".join(rng.choice(list("ACGT"), size=70))))
        ns.append(round(len(tr) / len(motif)))
    ns = np.array(ns)
    eng = sb.Engine()
    tab, off = eng.ref_boundary_tables(families_to_batch(fams), ns - 1, ns + 1)
    for i, (motif, tr, fl, fr) in enumerate(fams):
        ref_size = len(tr)
        for n in range(int(ns[i]) - 1, int(ns[i]) + 2):
            (ofs, ora), (ors, ola) = oracle.score_ref_boundaries(tr, fl, fr, motif, n, ref_size)
            fs, fe, rs, re = (int(v) for v in tab[int(off[i]) + n - int(ns[i]) + 1])
            assert (fs, fe + 1 - len(fl) - ref_size) == (ofs, ora)
            assert (rs, re + 1 - len(fr) - ref_size) == (ors, ola)
    eng.close()


def test_ref_boundary_tables_golden(sb, oracle, golden):
    """Both kernels pinned to the golden vectors: the packed kernel in reference mode (KERNEL_AUTO) and the general
    kernel's ARGMAX sweeps."""
    eng = sb.Engine()
    fams = [(c["motif"], c["tr_seq"], c["flank_left_seq"], c["flank_right_seq"]) for c in golden["boundaries"]]
    ns = np.array([c["n"] for c in golden["boundaries"]])
    lo = np.maximum(ns - 2, np.array([0 if (f[2] and f[3]) else 1 for f in fams]))
    hi = ns + 2
    for kernel in (sb.KERNEL_AUTO, sb.KERNEL_GENERAL):
        tab, off = eng.ref_boundary_tables(families_to_batch(fams), lo, hi, kernel=kernel)
        st = eng.stats()
        assert st["reads_packed_kernel"] + st["reads_general_kernel"] == len(fams)
        assert (st["reads_packed_kernel"] > 0) == (kernel == sb.KERNEL_AUTO)
        for i, c in enumerate(golden["boundaries"]):
            fs, fe, rs, re = (int(v) for v in tab[int(off[i]) + c["n"] - int(lo[i])])
            r_adj = fe + 1 - len(c["flank_left_seq"]) - c["ref_size"]
            l_adj = re + 1 - len(c["flank_right_seq"]) - c["ref_size"]
            assert [fs, r_adj, rs, l_adj] == c["expect"], (kernel, c)
            for n in range(int(lo[i]), int(hi[i]) + 1):  # the rest of the window against the oracle
                (ofs, ora), (ors, ola) = oracle.score_ref_boundaries(c["tr_seq"], c["flank_left_seq"],
                                                                     c["flank_right_seq"], c["motif"], n, c["ref_size"])
                fs, fe, rs, re = (int(v) for v in tab[int(off[i]) + n - int(lo[i])])
                assert (fs, fe + 1 - len(c["flank_left_seq"]) - c["ref_size"]) == (ofs, ora), (kernel, c, n)
                assert (rs, re + 1 - len(c["flank_right_seq"]) - c["ref_size"]) == (ors, ola), (kernel, c, n)


def test_invalid_inputs_raise(sb):
    from strkit_b200._native import StrkError

    eng = sb.Engine()
    p = sb.RepeatCountParams("repalign", 50, 3, 1)
    with pytest.raises(StrkError):
        eng.count_reads(families_to_batch([("CAG", "", "", "")], est=[0]), p)  # empty db
    b = families_to_batch([("CAG", "CAGCAG", "AC", "GT")])
    b.motif_len[0] = 0
    with pytest.raises(StrkError):
        eng.count_reads(b, p)
    b = families_to_batch([("CAG", "CAGCAG" * 40, "AC", "GT")] * 600, est=[40] * 599 + [1 << 23])   # garbage estimate
    with pytest.raises(StrkError, match="est_cn"):
        eng.count_reads(b, p)                     # (device-side planning: more than 512 reads)
    with pytest.raises(StrkError, match="est_cn"):
        eng.count_reads(families_to_batch([("CAGCAG", "CAGCAG", "AC", "GT")], est=[(1 << 22) - 1]), p)  # m * est > 2^24
    b = families_to_batch([("CAG", "CAGCAG", "AC", "GT")])
    b.seq_off[0] = np.uint64(2 ** 64 - 4)        # offset + length wraps around 64 bits
    with pytest.raises(StrkError, match="arena"):
        eng.count_reads(b, p)
    with pytest.raises(StrkError):
        sb.Engine(gap_open=7, gap_extend=1)  # affine gaps are not what the reference uses
    with pytest.raises(NotImplementedError):
        sb.get_repeat_count(3, "CAGCAG", "A", "T", "CAG", sb.RepeatCountParams("comp", 50, 3, 1))


def test_get_ref_repeat_count_golden(sb, golden):
    """Drop-in get_ref_repeat_count against vectors produced by the reference's own repeats.py:73-192."""
    for c in golden["ref"]:
        e = c["expect"]
        params = sb.RepeatCountParams("repalign", c["max_iters"], c["local_search_range"], c["step_size"])
        res = sb.get_ref_repeat_count(c["start_count"], c["tr_seq"], c["flank_left_seq"], c["flank_right_seq"],
                                      c["motif"], c["ref_size"], c["vcf_anchor_size"], params, c["respect_coords"])
        (cn, score), lo, ro, (n_off, n_fin), (fl2, tr2, fr2) = res
        assert (cn, score, lo, ro, n_off, n_fin) == (e["cn"], e["score"], e["l_offset"], e["r_offset"],
                                                     e["n_offset_scores"], e["n_iters_final"]), c
        assert (fl2, tr2, fr2) == (e["fl"], e["tr"], e["fr"])


def test_ref_counts_batch_with_reference_tiers(sb, oracle):
    """One C-ABI call for many loci, search parameters tiered like repeat_count_params.py:17-42
    (steps of 3 / 5 / 15 for large reference tracts), then the same loci one call per tier, with start counts off by
    tens of copies that send searches out of their first window (the device-side second look and the loci finished on
    the host)."""
    rng = np.random.default_rng(21)
    fams, starts, ref_sizes, rcs = [], [], [], []
    for i in range(40):
        m = int(rng.integers(2, 7))
        motif = "".join(rng.choice(list("ACGT"), size=m))
        k = int(rng.choice([12, 30, 80, 210, 450])) if i % 4 else int(rng.integers(5, 40))
        tr = mutate(rng, motif * k, 0.01, 0.005, 0.005)
        fl = "".join(rng.choice(list("ACGT"), size=70))
        fr = "".join(rng.choice(list("ACGT"), size=70))
        if i % 3 == 0:  # repeat spills into the flanks
            fl = fl[:60] + (motif * 10)[-10:]
            fr = (motif * 10)[:8] + fr[8:]
        est = round(len(tr) / m)
        p = sb.get_reference_rc_params("repalign", est * (10 if i % 5 == 0 else 1), 250)  # exercise every tier
        fams.append((motif, tr, fl, fr))
        starts.append(est)
        ref_sizes.append(len(tr))
        rcs.append([p.max_iters, p.initial_local_search_range, p.initial_step_size])
    eng = sb.Engine()
    got = eng.ref_counts(families_to_batch(fams), starts, ref_sizes, np.array(rcs), vcf_anchor_size=5)
    for i, (motif, tr, fl, fr) in enumerate(fams):
        (cn, score), lo, ro, (n_off, n_fin), (fl2, tr2, fr2) = oracle.get_ref_repeat_count(
            starts[i], tr, fl, fr, motif, ref_sizes[i], 5, rcs[i][0], rcs[i][1], rcs[i][2])
        assert got[i].tolist() == [cn, score, lo, ro, n_off, n_fin, len(fl2), len(fr2)], (i, fams[i][0], rcs[i])
    starts = np.array(starts)
    bad = rng.random(starts.shape[0]) < 0.2
    starts[bad] = np.maximum(0, starts[bad] + rng.integers(-30, 60, int(bad.sum())))
    redone = 0
    for tier in sorted({tuple(r) for r in rcs}):
        idx = [i for i, r in enumerate(rcs) if tuple(r) == tier]
        got = eng.ref_counts(families_to_batch([fams[i] for i in idx]), starts[idx], [ref_sizes[i] for i in idx],
                             np.array([rcs[i] for i in idx]), vcf_anchor_size=5)
        redone += int(eng.stats()["widening_passes"])
        for row, i in zip(got, idx):
            motif, tr, fl, fr = fams[i]
            (cn, score), lo, ro, (n_off, n_fin), (fl2, tr2, fr2) = oracle.get_ref_repeat_count(
                int(starts[i]), tr, fl, fr, motif, ref_sizes[i], 5, *tier)
            assert row.tolist() == [cn, score, lo, ro, n_off, n_fin, len(fl2), len(fr2)], (i, motif, tier, starts[i])
    assert redone > 0   # some searches did leave their first window


def test_ragged_loci_zero_one_and_max_reads(sb, oracle):
    """Loci with 0, 1, 3 and 250 reads (the reference caps a locus at max_reads = 250, params.py:21) in one batch;
    the carried start offset of call_locus.py:1129-1161 runs over every read of the 250-read locus."""
    from strkit_b200.batcher import LocusReads, pack_loci
    from tests.helpers import mutate, rand_seq

    rng = np.random.default_rng(21)
    loci = []
    for n_reads in (0, 1, 250, 3, 0, 17):
        m = int(rng.integers(2, 7))
        motif = rand_seq(rng, m)
        k = int(rng.integers(8, 30))
        fl, fr = rand_seq(rng, 70), rand_seq(rng, 70)
        trs, fls, frs, est = [], [], [], []
        for _ in range(n_reads):
            kk = k + int(rng.choice([-2, -1, 0, 0, 0, 1, 2]))
            tr = mutate(rng, motif * kk, 0.01, 0.01, 0.01)
            trs.append(tr or motif)
            fls.append(mutate(rng, fl, 0.01, 0.0, 0.0)[-70:] or "A")
            frs.append(mutate(rng, fr, 0.01, 0.0, 0.0)[:70] or "A")
            est.append(round(len(trs[-1]) / m))
        loci.append(LocusReads(motif, est, trs, fls, frs))
    batch = pack_loci(loci)
    assert np.diff(batch.read_begin).tolist() == [0, 1, 250, 3, 0, 17]
    params = sb.RepeatCountParams("repalign", 50, 3, 1)
    eng = sb.Engine()
    got = eng.count_reads(batch, params)
    want, _ = oracle.count_loci(batch.arena, batch.seq_off, batch.lens, batch.est_cn, batch.read_begin, batch.motif_off,
                                batch.motif_len, n_threads=8)
    assert np.array_equal(got, want), np.flatnonzero((got != want).any(axis=1))[:10]
    eng.close()


def test_full_size_catalog_properties(sb, oracle):
    """BASELINE config 2 at its full size: 1 048 576 loci x 30 reads (31.5 M reads), streamed as 32 768-locus
    blocks.  Size-independent checks: (i) bit-exact parity with the CPU oracle on loci sampled from blocks spread over
    the whole catalog; (ii) results do not depend on how the catalog is cut into blocks; (iii) invariants of every
    read: score <= 2 * |db| (match = 2), 1 <= n_explored <= max_iters + 2 * range + 1, the reported start within the
    carried-offset range of its estimate; (iv) the count equals the number of copies written into the read for the
    overwhelming majority of (HiFi-like) reads."""
    import torch

    from strkit_b200 import synth

    n_blocks, block = 32, 32768
    params = sb.RepeatCountParams("repalign", 50, 3, 1)
    eng = sb.Engine()
    rng = np.random.default_rng(4)
    cut_blocks = set(rng.choice(n_blocks, size=3, replace=False).tolist())
    oracle.set_simd(True)   # the AVX2 alignments of the CPU port: asserted identical to the scalar ones (test_oracle_golden)

    def blocks():
        for i in range(n_blocks):
            sbatch = synth.generate(synth.CONFIGS[2], block, seed=910_000 + i, device="cuda", chunk_loci=4096)
            hb = sbatch.to_host(pin=True, nibble=True)     # what the batcher ships: nibble-packed arenas
            hb.true_cn = sbatch.true_cn.cpu().numpy()
            lo = int(rng.integers(0, block - 256))
            hb.check = (lo, sbatch.to_host().slice_loci(lo, lo + 256, compact=True))   # 256 loci of EVERY block
            del sbatch
            yield hb

    n_reads = n_equal = n_checked = 0

    def tee():
        for i, hb in enumerate(blocks()):
            stash.append((i, hb))
            yield hb

    stash: list = []
    kept = {}
    for out in eng.count_reads_stream(tee(), params):
        i, hb = stash.pop(0)
        db_len = hb.lens.sum(axis=1)
        assert (out[:, 1] <= 2 * db_len).all() and (out[:, 0] >= 0).all()
        assert (out[:, 2] >= 1).all() and (out[:, 2] <= 50 + 2 * 3 + 1).all()
        assert (np.abs(out[:, 3] - hb.est_cn) <= 64).all()
        n_reads += out.shape[0]
        n_equal += int((out[:, 0] == hb.true_cn).sum())
        lo, sub = hb.check
        want, _ = oracle.count_loci(sub.arena, sub.seq_off, sub.lens, sub.est_cn, sub.read_begin, sub.motif_off,
                                    sub.motif_len, n_threads=16)
        r0, r1 = int(hb.read_begin[lo]), int(hb.read_begin[lo + 256])
        assert np.array_equal(out[r0:r1], want), (i, lo)
        n_checked += r1 - r0
        if i in cut_blocks:
            kept[i] = (hb, out.copy())
    oracle.set_simd(False)
    assert n_reads == n_blocks * block * 30 and n_checked == n_blocks * 256 * 30   # 245 760 reads against the CPU port
    assert n_equal / n_reads > 0.97
    torch.cuda.empty_cache()
    for i, (hb, out) in sorted(kept.items()):
        # a different cut of the same loci gives the same rows
        cut = int(rng.integers(1, block - 1))
        a, b = hb.slice_loci(0, cut), hb.slice_loci(cut, block)
        again = np.concatenate(list(eng.count_reads_stream([a, b], params)))
        assert np.array_equal(again, out), (i, cut)


def test_nibble_arenas_equal_ascii(sb, oracle):
    """STRK_ARENA_NIBBLE: the nibble-packed host arena (half the H2D bytes) gives the rows of the ASCII one -- blocking
    call, streamed blocks, resident batch; wildcards, lower case (folded by the packer), odd offsets, tiny batches."""
    from strkit_b200 import synth
    from strkit_b200.batcher import LocusReads, pack_loci

    params = sb.RepeatCountParams("repalign", 50, 3, 1)
    eng = sb.Engine()
    for cfg, n in ((2, 2000), (3, 700)):
        b = synth.generate(synth.CONFIGS[cfg], n, seed=60 + cfg).to_host()
        want = eng.count_reads(b, params)
        nb = b.to_nibble()
        assert nb.arena.nbytes * 2 - b.arena.nbytes in (0, 1)
        assert np.array_equal(eng.count_reads(nb, params), want)
        halves = [nb.slice_loci(0, n // 3), nb.slice_loci(n // 3, n)]
        assert np.array_equal(np.concatenate(list(eng.count_reads_stream(halves, params))), want)
        db = eng.upload(nb)
        eng.run(db, params)
        assert np.array_equal(eng.download(db), want)
        db.free()
    rng = np.random.default_rng(3)
    loci = [LocusReads("CAG", [4, 5], ["cagCAGXAGCAGC", "CAGCAGNAGCAGCAG"], ["ACGTT", "acgtt"], ["TTGAC", "TTGA"]),
            LocusReads("AT", [3], ["ATATAT"], ["G"], ["C"])]
    a, nb = pack_loci(loci), pack_loci(loci, nibble=True)
    assert nb.arena_format == 1
    got_a, got_n = eng.count_reads(a, params), eng.count_reads(nb, params)
    want, _ = oracle.count_loci(a.arena, a.seq_off, a.lens, a.est_cn, a.read_begin, a.motif_off, a.motif_len)
    assert np.array_equal(got_a, want) and np.array_equal(got_n, want)
    eng.close()


def test_rust_ext_shaped_entry_point(sb, oracle):
    """strk_get_repeat_count / strkit_rust_ext_shim.get_repeat_count: the 9-argument PyO3 signature of repeats.py:58-68."""
    from strkit_b200.strkit_rust_ext_shim import get_repeat_count as rust_shaped

    rng = np.random.default_rng(31)
    for i, (motif, tr, fl, fr) in enumerate(random_families(rng, 60, max_k=30, flank_choices=(5, 20, 70))):
        start = max(0, round(len(tr) / len(motif)) + int(rng.integers(-4, 5)))
        mi, r_, st = [(50, 3, 1), (250, 3, 1), (30, 5, 2), (8, 1, 3)][i % 4]
        assert rust_shaped(start, tr, fl, fr, motif, mi, r_, st) == oracle.get_repeat_count(start, tr, fl, fr, motif, mi, r_, st)
        assert rust_shaped(start, tr, fl, fr, motif, mi, r_, st, use_shortcuts=False)[1] >= 1
    with pytest.raises(NotImplementedError):
        rust_shaped(5, "CAGCAG", "AC", "GT", "CAG", 50, 3, 1, use_shortcuts=True)


def test_block_session_equals_per_call_loop(sb, oracle):
    """Block mode on the GPU: one BlockSession.run() for a block of loci, then the reference's read loop (restated with
    shims in tests/ref_loop_shim.py) bound to its look-ups, against the same loop making one GPU call per read and
    against the CPU port: identical read dictionaries and log lines, zero cache misses."""
    from tests.test_host_cpu import make_block_loci, run_block_vs_per_call

    p = sb.RepeatCountParams("repalign", 50, 3, 1)
    loci = make_block_loci(seed=9, n_loci=40)
    sb.get_repeat_count.cache_clear()
    run_block_vs_per_call(loci, sb.default_engine(), sb.get_repeat_count, p)

    def cpu(start_count, tr_seq, flank_left_seq, flank_right_seq, motif, rc_params):
        return oracle.get_repeat_count(start_count, tr_seq, flank_left_seq, flank_right_seq, motif, rc_params.max_iters,
                                       rc_params.initial_local_search_range, rc_params.initial_step_size)

    session = run_block_vs_per_call(loci, sb.default_engine(), cpu, p)
    # reference windows through the same session
    rp = sb.get_reference_rc_params("repalign", 20, 250)
    args = (20, "CAG" * 20, "ACGTTGCATGCATTGACCATGACTGAATCG", "TTGACGATCGGATCGATTAGCTAGCTAAGC", "CAG", 60, 5, rp)
    session.add_reference(*args)
    session.run()
    want = oracle.get_ref_repeat_count(*args[:7], rp.max_iters, rp.initial_local_search_range, rp.initial_step_size)
    assert session.get_ref_repeat_count(*args) == want and session.ref_misses == 0


def test_stream_with_reference_windows(sb):
    """count_reads_stream(refs=...): a block's reference windows ride in the same run phase; rows equal the separate calls."""
    from bench import ref_windows_of
    from strkit_b200 import synth

    params = sb.RepeatCountParams("repalign", 50, 3, 1)
    eng = sb.Engine()
    blocks = [synth.generate(synth.CONFIGS[2], 900, seed=70 + i).to_host() for i in range(3)]
    refs = [ref_windows_of(b, np) for b in blocks]
    want_reads = [eng.count_reads(b, params) for b in blocks]
    want_refs = [eng.ref_counts(r[0], r[1], r[2], r[3], r[4]) for r in refs]
    st = eng.stats()
    assert st["executed_cells"] > 0 and st["dp_ms"] > 0          # strk_ref_counts reports its own counters
    got = list(eng.count_reads_stream([b.to_nibble() for b in blocks], params, refs=refs))
    for (reads, ref_out), wr, wf in zip(got, want_reads, want_refs):
        assert np.array_equal(reads, wr) and np.array_equal(ref_out, wf)
    eng.close()


def test_config4_to_spec_full_search(sb, oracle):
    """BASELINE config 4 as SURVEY 8d specifies it: motifs of catalogs/pathogenic_assoc.hg38.tsv (IUPAC ones included,
    reads synthesised with the reference's own IUPAC table), tracts of 3-6 kb, the FULL search of count_reads (not +-1
    tables) and get_ref_repeat_count with the reference's tiers for large tracts (steps 3 / 5 / 15,
    repeat_count_params.py:25-35), against the CPU port (AVX2 alignments, asserted identical to the scalar ones)."""
    from strkit_b200 import synth

    assert len(synth.PATHOGENIC_MOTIFS) == 44 and synth.IUPAC_BASES["D"] == "ACT"
    motifs = ["RAAAT", "GCN", "AARRG", "CASR", "GCCCCG", "GCGCGGGGCGGG", "CAG", "TRRAA"]
    batch, loci = synth.generate_expansions(n_loci=8, reads_per_locus=5, seed=77, max_tract=6000, big_lo=600, big_hi=2000,
                                            motifs=motifs)
    tract = batch.lens[:, 1]
    assert tract.max() > 5500 and (tract > 3000).sum() >= 10
    params = sb.RepeatCountParams("repalign", 50, 3, 1)
    eng = sb.Engine()
    oracle.set_simd(True)
    try:
        got = eng.count_reads(batch, params)
        want, _ = oracle.count_loci(batch.arena, batch.seq_off, batch.lens, batch.est_cn, batch.read_begin, batch.motif_off,
                                    batch.motif_len, n_threads=16)
        assert np.array_equal(got, want), np.flatnonzero((got != want).any(axis=1))[:10]
        assert eng.stats()["reads_general_kernel"] >= 10
        # reference windows: the longest read of each of 5 loci stands in for the reference genome, tiers by copy number
        fams, starts, sizes, rcs = [], [], [], []
        for lr in loci[:5]:
            k = int(np.argmax([len(t) for t in lr.tr_seqs]))
            tr, fl, fr = lr.tr_seqs[k], lr.flank_left_seqs[k], lr.flank_right_seqs[k]
            est = round(len(tr) / len(lr.motif))
            p = sb.get_reference_rc_params("repalign", est, 250)
            fams.append((lr.motif, tr, fl, fr))
            starts.append(est)
            sizes.append(len(tr))
            rcs.append([p.max_iters, p.initial_local_search_range, p.initial_step_size])
        assert {r[2] for r in rcs} >= {3, 5}      # large-tract tiers exercised
        rcs[0] = [50, 1, 15]                      # the >= 2000-copy tier (a 6 kb tract holds at most 2000 3-mers)
        got = eng.ref_counts(families_to_batch(fams), starts, sizes, np.array(rcs), vcf_anchor_size=5)
        for i, (motif, tr, fl, fr) in enumerate(fams):
            (cn, score), lo, ro, (n_off, n_fin), (fl2, _, fr2) = oracle.get_ref_repeat_count(
                starts[i], tr, fl, fr, motif, sizes[i], 5, rcs[i][0], rcs[i][1], rcs[i][2])
            assert got[i].tolist() == [cn, score, lo, ro, n_off, n_fin, len(fl2), len(fr2)], (i, motif, rcs[i])
    finally:
        oracle.set_simd(False)
    eng.close()
