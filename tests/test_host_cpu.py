"""CPU-side tests (no GPU): the C-ABI library loads and exports what include/strkit_b200.h declares,
fails loudly without a device, and the host batcher / generators behave."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from strkit_b200 import _native

    header = open(os.path.join(ROOT, "include", "strkit_b200.h")).read()
    declared = set(re.findall(r"\b(strk_[a-z_0-9]+)\s*\(", header))
    assert len(declared) >= 15
    raw = ctypes.CDLL(_native.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(raw, name), f"{name} declared in the header but not exported"
    assert declared == set(_native.EXPORTED)
    assert _native.lib.strk_version().decode().startswith("strkit_b200")


def test_no_cpu_fallback_without_device():
    import strkit_b200
    from strkit_b200._native import StrkError

    if strkit_b200.device_count() > 0:
        pytest.skip("a GPU is visible")
    with pytest.raises(StrkError, match="no CPU fallback"):
        strkit_b200.Engine()
    with pytest.raises(StrkError):
        strkit_b200.get_repeat_count(5, "CAGCAGCAGCAGCAG", "ACGT", "TTGA", "CAG",
                                     strkit_b200.RepeatCountParams("repalign", 50, 3, 1))


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "strkit_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.lower(), f"{f} mentions the oracle"


def test_matrix_matches_reference_golden(golden):
    from strkit_b200.align_matrix import dna_bases_str, dna_matrix

    assert dna_bases_str == golden["alphabet"]
    assert dna_matrix.tolist() == golden["matrix"]


def test_reference_rc_param_tiers():
    from strkit_b200 import get_reference_rc_params as g

    assert (g("repalign", 10, 250).max_iters, g("repalign", 10, 250).initial_step_size) == (250, 1)
    p = g("repalign", 200, 250)
    assert (p.max_iters, p.initial_step_size, p.initial_local_search_range) == (200, 3, 3)
    p = g("repalign", 1999, 250)
    assert (p.max_iters, p.initial_step_size, p.initial_local_search_range) == (150, 5, 3)
    p = g("repalign", 2000, 250)
    assert (p.max_iters, p.initial_step_size, p.initial_local_search_range) == (50, 15, 1)


def test_pack_loci_layout():
    from strkit_b200 import LocusReads, pack_loci

    b = pack_loci([LocusReads("CAG", [2, 3], ["CAGCAG", "CAGCAGCAG"], ["AA", "AC"], ["TT", "T"]),
                   LocusReads("AT", [1], ["AT"], [""], ["GG"])])
    b.validate()
    assert b.n_reads == 3 and b.n_loci == 2
    assert b.read_begin.tolist() == [0, 2, 3]
    assert b.lens.tolist() == [[2, 6, 2], [2, 9, 1], [0, 2, 2]]
    arena = bytes(b.arena)
    assert arena[int(b.seq_off[1]):int(b.seq_off[1]) + 12] == b"ACCAGCAGCAGT"
    assert arena[int(b.motif_off[1]):int(b.motif_off[1]) + 2] == b"AT"
    s = b.slice_loci(1, 2)
    assert s.n_reads == 1 and s.read_begin.tolist() == [0, 1] and s.lens.tolist() == [[0, 2, 2]]


def test_pack_loci_c_helper_equals_python_body():
    """csrc/fastpack.c (built by __graft_entry__.build()) and the pure-Python body of pack_loci produce the same
    arrays: ragged loci, empty strings, a locus without reads, tuples instead of lists, numpy estimates."""
    import importlib

    import __graft_entry__
    from strkit_b200 import LocusReads, batcher
    from tests.helpers import random_families

    if batcher._fastpack is None:  # first run in a fresh tree
        __graft_entry__.build()
        importlib.reload(batcher)
    if batcher._fastpack is None:
        pytest.skip("no Python.h / C compiler on this box: _fastpack.so cannot be built")
    pack_loci = batcher.pack_loci
    rng = np.random.default_rng(9)
    fams = random_families(rng, 300)
    loci, at = [], 0
    while at < len(fams):
        n = int(rng.integers(0, 6))
        grp = fams[at:at + n]
        at += n
        motif = grp[0][0] if grp else "ACG"
        loci.append(LocusReads(motif, np.array([len(t) // len(motif) for _, t, _, _ in grp], dtype=np.int64),
                               tuple(t for _, t, _, _ in grp), [fl for _, _, fl, _ in grp], [fr for _, _, _, fr in grp]))
    for subset in (loci, loci[:1], []):
        a, b = pack_loci(subset, use_helper=True), pack_loci(subset, use_helper=False)
        for f in ("arena", "seq_off", "lens", "est_cn", "read_begin", "motif_off", "motif_len"):
            x, y = getattr(a, f), getattr(b, f)
            assert x.dtype == y.dtype and x.shape == y.shape and np.array_equal(x, y), f
        a.validate()
    with pytest.raises(ValueError):
        pack_loci([LocusReads("AC", [1], ["AC\u00e9"], ["A"], ["C"])])
    with pytest.raises(ValueError):
        pack_loci([LocusReads("AC", [1, 2], ["AC"], ["A"], ["C"])])


def test_synth_generator_is_deterministic_and_sane(oracle):
    from strkit_b200 import synth

    a = synth.generate(synth.CONFIGS[1], 50, seed=1).to_host()
    b = synth.generate(synth.CONFIGS[1], 50, seed=1).to_host()
    assert np.array_equal(a.arena, b.arena) and np.array_equal(a.lens, b.lens)
    assert a.n_reads == 1500 and (a.lens[:, 0] <= 70).all() and (a.lens[:, 2] <= 70).all()
    assert set(np.unique(a.arena)) <= set(b"ACGTX")
    # the generator's copies are recovered by the reference search on almost every HiFi read
    sb = synth.generate(synth.CONFIGS[1], 50, seed=1)
    out, _ = oracle.count_loci(a.arena, a.seq_off, a.lens, a.est_cn, a.read_begin, a.motif_off, a.motif_len,
                               n_threads=4)
    assert (out[:, 0] == sb.true_cn.numpy()).mean() > 0.97


def test_install_rebinds_strkit_names(monkeypatch):
    """install() must patch both strkit.call.repeats and the from-imported names in strkit.call.call_locus
    (call_locus.py:32).  Uses stand-in modules: the real strkit is not installable in the test box."""
    import sys
    import types

    import strkit_b200
    from strkit_b200 import repeats as ours

    pkg, call = types.ModuleType("strkit"), types.ModuleType("strkit.call")
    rep, loc = types.ModuleType("strkit.call.repeats"), types.ModuleType("strkit.call.call_locus")
    rep.get_repeat_count = rep.get_ref_repeat_count = lambda *a, **k: "reference"
    loc.get_repeat_count, loc.get_ref_repeat_count = rep.get_repeat_count, rep.get_ref_repeat_count
    for name, mod in (("strkit", pkg), ("strkit.call", call), ("strkit.call.repeats", rep),
                      ("strkit.call.call_locus", loc)):
        monkeypatch.setitem(sys.modules, name, mod)
    patched = strkit_b200.install()
    assert len(patched) == 4
    assert loc.get_repeat_count is ours.get_repeat_count and rep.get_ref_repeat_count is ours.get_ref_repeat_count
    strkit_b200.uninstall()
    assert loc.get_repeat_count() == "reference" and rep.get_ref_repeat_count() == "reference"
    # opt-in: call_alleles (allele.py:176, from-imported at call_locus.py:28)
    al = types.ModuleType("strkit.call.allele")
    al.call_alleles = loc.call_alleles = lambda *a, **k: "reference"
    monkeypatch.setitem(sys.modules, "strkit.call.allele", al)
    assert len(strkit_b200.install()) == 4 and loc.call_alleles() == "reference"
    strkit_b200.uninstall()
    patched = strkit_b200.install(alleles=True)
    assert len(patched) == 6 and loc.call_alleles is strkit_b200.call_alleles and al.call_alleles is strkit_b200.call_alleles
    strkit_b200.uninstall()
    assert loc.call_alleles() == "reference" and al.call_alleles() == "reference"


def test_bench_reference_arm_prints_one_contract_line():
    """bench.py --impl reference (the CPU arm the driver runs next to ours): one JSON line on stdout with the
    contract's keys, exactly K timed steps; ranks other than 0 print nothing."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
           "--cpu-sample-loci", "48"]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    out = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stderr[-500:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["steps"] == 2 and d["warmup"] == 1 and d["higher_is_better"] is True
    for key in ("metric", "value", "unit", "n_gpus", "ms_per_step", "scaling", "vs_baseline", "dtype", "data"):
        assert key in d, key
    assert "workload" in d["config"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    out = subprocess.run(cmd, capture_output=True, text=True, env=dict(env, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1"),
                         timeout=600)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_bench_strong_scaling_line_is_json(monkeypatch):
    """bench.py --scaling strong needs GPUs to run, but the line it prints is assembled by a pure function: numpy
    scalars in (what the run produces), one json.dumps-able dict with the contract's keys out."""
    import importlib
    import json
    import sys

    monkeypatch.setattr(sys, "argv", ["bench.py", "--gpus", "2", "--steps", "32", "--warmup", "3", "--scaling", "strong"])
    bench = importlib.import_module("bench")
    args = bench.parse_args()
    line = bench.strong_scaling_line(args, 2, 32, 32768, np.int64(32 * 32768 * 30), np.float64(0.27),
                                     [np.float64(0.26), np.float64(0.27)], [np.int64(524165), np.int64(524411)], np.int64(32768),
                                     np.int64(86_000_000), np.int64(15_700_000), np.int64(828), np.bool_(True),
                                     {"sm_mhz": 1965.0, "sm_max_mhz": 1965.0, "reasons": []}, None)
    d = json.loads(json.dumps(line))
    assert d["scaling"] == "strong" and d["n_gpus"] == 2 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["value"] == d["e2e"]["value"] == pytest.approx(32 * 32768 * 30 / 0.27)
    assert d["partition"]["loci_per_rank"] == [524165, 524411] and d["partition"]["loci_per_streamed_block"] == 32768
    assert d["partition"]["imbalance_max_over_mean"] == pytest.approx(0.27 / 0.265)
    for key in ("metric", "unit", "steps", "warmup", "ms_per_step", "dtype", "data", "config", "gpu_launches", "clocks"):
        assert key in d, key
    assert "workload" in d["config"]


def test_bench_dump_outputs_exact_and_capped(monkeypatch, tmp_path):
    """bench.py --dump-outputs: int32 results land as float64 without loss; above the size cap every array keeps the
    same seeded sample of its rows, identical from call to call; the flag is refused outside the default workload."""
    import importlib
    import sys

    bench = importlib.import_module("bench")
    rng = np.random.default_rng(3)
    reads = rng.integers(-2**31, 2**31 - 1, size=(3000, 4), dtype=np.int64).astype(np.int32)
    ref = rng.integers(-2**31, 2**31 - 1, size=(100, 8), dtype=np.int64).astype(np.int32)
    bench.dump_outputs(str(tmp_path / "full"), {"read_counts": reads, "ref_counts": ref})
    for name, a in (("read_counts", reads), ("ref_counts", ref)):
        got = np.load(tmp_path / "full" / f"{name}.npy")
        assert got.dtype == np.float64 and np.array_equal(got.astype(np.int32), a)
    limit = (3000 * 4 + 100 * 8) * 8 // 4
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"read_counts": reads, "ref_counts": ref}, limit=limit)
    a, b = (np.load(tmp_path / d / "read_counts.npy") for d in ("a", "b"))
    assert a.shape == (750, 4) and np.array_equal(a, b)
    rows = {tuple(r) for r in reads.tolist()}
    assert all(tuple(int(v) for v in row) in rows for row in a)
    assert sum((tmp_path / "a" / f).stat().st_size - 128 for f in ("read_counts.npy", "ref_counts.npy")) <= limit
    monkeypatch.setattr(sys, "argv", ["bench.py", "--config", "3", "--dump-outputs", str(tmp_path / "x")])
    with pytest.raises(SystemExit):
        bench.parse_args()


# ---------------------------------------------------------------------------------------------------------------
# host batcher: nibble arenas, compact slices, the C packing helper
# ---------------------------------------------------------------------------------------------------------------
def _decode(b, off, n):
    from strkit_b200.batcher import ARENA_NIBBLE

    if b.arena_format == ARENA_NIBBLE:
        idx = np.arange(off, off + n)
        byte = b.arena[idx >> 1]
        return "".join("ACGTRYSWKMBDHVNX"[c] for c in np.where(idx & 1, byte >> 4, byte & 15))
    return bytes(b.arena[off:off + n]).decode()


def test_pack_loci_layouts_agree():
    """ASCII / nibble, C helper (1 and 3 copy threads) / pure-Python body, str / bytes inputs: the same reads."""
    from strkit_b200.batcher import LocusReads, pack_loci

    rng = np.random.default_rng(0)
    loci = []
    for l in range(300):
        m = int(rng.integers(1, 7))
        n = int(rng.integers(0, 6))
        trs = ["".join(rng.choice(list("ACGTXacgtn"), size=int(rng.integers(0, 40)))) for _ in range(n)]
        fls = ["".join(rng.choice(list("ACGT"), size=int(rng.integers(0, 9)))) for _ in range(n)]
        frs = ["".join(rng.choice(list("ACGT"), size=int(rng.integers(0, 9)))) for _ in range(n)]
        if l % 3 == 0:
            trs = [t.encode() for t in trs]
        loci.append(LocusReads("".join(rng.choice(list("ACGTN"), size=m)), [int(rng.integers(0, 30)) for _ in range(n)],
                               trs, fls, frs))
    a, p = pack_loci(loci), pack_loci(loci, use_helper=False)
    for f in ("arena", "seq_off", "lens", "est_cn", "read_begin", "motif_off", "motif_len"):
        assert np.array_equal(getattr(a, f), getattr(p, f)), f
    variants = [a, pack_loci(loci, nibble=True, threads=3), pack_loci(loci, nibble=True, threads=1),
                pack_loci(loci, use_helper=False, nibble=True), a.to_nibble(), a.to_nibble().to_ascii()]
    assert [v.arena_format for v in variants] == [0, 1, 1, 1, 1, 0]
    r = 0
    for l, lr in enumerate(loci):
        for v in variants:
            assert _decode(v, int(v.motif_off[l]), int(v.motif_len[l])).upper() == lr.motif.upper()
        for tr, fl, fr in zip(lr.tr_seqs, lr.flank_left_seqs, lr.flank_right_seqs):
            want = fl + (tr.decode() if isinstance(tr, bytes) else tr) + fr
            for v in variants:
                assert v.lens[r].tolist() == [len(fl), len(tr), len(fr)]
                assert _decode(v, int(v.seq_off[r]), len(want)).upper() == want.upper()
            r += 1
    # a byte outside the 16-letter alphabet has no nibble code: the block stays ASCII
    assert pack_loci([LocusReads("CAG", [3], ["CAG-AG"], ["AC"], ["GT"])], nibble=True).arena_format == 0
    with pytest.raises(ValueError):
        pack_loci([LocusReads("CAG", [3], ["CAG-AG"], ["AC"], ["GT"])]).to_nibble()


def test_pack_loci_threaded_walk_equals_single_thread():
    """Enough reads that the helper really splits the walk over its threads (one per 4 096 reads at most): ranges of
    loci of uneven size, every output array identical to one thread and to the pure-Python body, both layouts; an
    error found by a worker thread (non-ASCII str, wrong type, byte without a nibble code) surfaces as the exception
    of the single-threaded path."""
    from strkit_b200 import batcher
    from strkit_b200.batcher import LocusReads, pack_loci

    if batcher._fastpack is None:
        pytest.skip("_fastpack.so not built")
    rng = np.random.default_rng(5)
    letters = np.frombuffer(b"ACGT", dtype=np.uint8)

    def seq(n):
        return letters[rng.integers(0, 4, n)].tobytes().decode()

    loci = []
    for l in range(700):
        n = int(rng.integers(0, 60))
        motif = seq(int(rng.integers(1, 7)))
        loci.append(LocusReads(motif, [int(rng.integers(0, 50)) for _ in range(n)],
                               [seq(int(rng.integers(0, 90))) for _ in range(n)], [seq(int(rng.integers(0, 12))) for _ in range(n)],
                               [seq(int(rng.integers(0, 12))) for _ in range(n)]))
    assert sum(len(x.tr_seqs) for x in loci) > 3 * 4096
    for nibble in (False, True):
        one = pack_loci(loci, nibble=nibble, threads=1)
        body = pack_loci(loci, nibble=nibble, use_helper=False)
        for threads in (2, 4, 7):
            many = pack_loci(loci, nibble=nibble, threads=threads)
            assert many.arena_format == one.arena_format == body.arena_format == int(nibble)
            for f in ("arena", "seq_off", "lens", "est_cn", "read_begin", "motif_off", "motif_len"):
                assert np.array_equal(getattr(many, f), getattr(one, f)), (f, threads, nibble)
                if not nibble:  # (the Python body's nibble layout packs reads back to back: compared read by read above)
                    assert np.array_equal(getattr(many, f), getattr(body, f)), (f, threads, nibble)
        one.validate()
    last = loci[-1]
    bad_ascii = loci[:-1] + [LocusReads(last.motif, [1], ["AC\u00e9"], ["A"], ["C"])]
    bad_type = loci[:-1] + [LocusReads(last.motif, [1], [17], ["A"], ["C"])]
    bad_code = loci[:-1] + [LocusReads(last.motif, [1], ["AC-T"], ["A"], ["C"])]
    for threads in (1, 4):
        with pytest.raises(ValueError):
            pack_loci(bad_ascii, threads=threads)
        with pytest.raises(TypeError):
            pack_loci(bad_type, threads=threads)
        assert pack_loci(bad_code, nibble=True, threads=threads).arena_format == 0  # falls back to the ASCII layout


def test_synth_nibble_and_compact_slices():
    from strkit_b200 import synth

    b = synth.generate(synth.CONFIGS[2], 60, seed=1).to_host()
    nb = synth.generate(synth.CONFIGS[2], 60, seed=1).to_host(nibble=True)
    assert nb.arena_format == 1 and np.array_equal(b.to_nibble().arena, nb.arena)
    assert np.array_equal(nb.to_ascii().arena[:b.arena.shape[0]], b.arena)
    full, cut = b.slice_loci(10, 25), b.slice_loci(10, 25, compact=True)
    assert cut.arena.nbytes < 0.4 * full.arena.nbytes
    for r in range(cut.n_reads):
        n = int(cut.lens[r].sum())
        assert _decode(cut, int(cut.seq_off[r]), n) == _decode(full, int(full.seq_off[r]), n)
    for l in range(cut.n_loci):
        assert _decode(cut, int(cut.motif_off[l]), int(cut.motif_len[l])) == _decode(full, int(full.motif_off[l]),
                                                                                     int(full.motif_len[l]))
    assert b.slice_loci(7, 7, compact=True).n_reads == 0


# ---------------------------------------------------------------------------------------------------------------
# block mode (strkit_b200.locus_block): host logic, with the device call replaced by the CPU checker
# ---------------------------------------------------------------------------------------------------------------
class _CheckerEngine:
    """Stands in for Engine in CPU tests of the HOST logic: the same calls, answered by the CPU checker."""

    def __init__(self, oracle):
        import threading

        self.oracle, self.lock, self.calls = oracle, threading.RLock(), 0

    def count_reads(self, batch, rc_params, kernel=0, out=None):
        self.calls += 1
        b = batch.to_ascii()
        return self.oracle.count_loci(b.arena, b.seq_off, b.lens, b.est_cn, b.read_begin, b.motif_off, b.motif_len,
                                      max_iters=rc_params.max_iters, local_search_range=rc_params.initial_local_search_range,
                                      step_size=rc_params.initial_step_size)[0]

    def ref_counts(self, batch, start_count, ref_size, rc, vcf_anchor_size, respect_coords=False):
        self.calls += 1
        arena = batch.arena.tobytes().decode()
        out = np.zeros((batch.n_loci, 8), dtype=np.int32)
        for l in range(batch.n_loci):
            o, (nfl, ntr, nfr) = int(batch.seq_off[l]), (int(v) for v in batch.lens[l])
            motif = arena[int(batch.motif_off[l]):int(batch.motif_off[l]) + int(batch.motif_len[l])]
            (cn, sc), lo, ro, (n_off, n_fin), (fl2, _, fr2) = self.oracle.get_ref_repeat_count(
                int(start_count[l]), arena[o + nfl:o + nfl + ntr], arena[o:o + nfl], arena[o + nfl + ntr:o + nfl + ntr + nfr],
                motif, int(ref_size[l]), vcf_anchor_size, int(rc[l][0]), int(rc[l][1]), int(rc[l][2]), respect_coords)
            out[l] = [cn, sc, lo, ro, n_off, n_fin, len(fl2), len(fr2)]
        return out


def make_block_loci(seed=5, n_loci=24):
    """Loci for the read-loop comparison: clean reads, reads whose estimate is off (carried offset), junk reads that
    fail the score filter (one locus with enough of them to be abandoned), a read that exhausts the iteration budget."""
    from tests.helpers import mutate, rand_seq
    from tests.ref_loop_shim import SegmentShim

    rng = np.random.default_rng(seed)
    loci = []
    for l in range(n_loci):
        m = int(rng.integers(2, 7))
        motif = rand_seq(rng, m)
        k = int(rng.integers(8, 40))
        fl, fr = rand_seq(rng, 90), rand_seq(rng, 90)
        segs = []
        for r in range(int(rng.integers(1, 14))):
            kk = max(1, k + int(rng.choice([-2, -1, 0, 0, 0, 1, 3])))
            tr = mutate(rng, motif * kk, 0.01, 0.01, 0.01) or motif
            if l % 6 == 1 and r % 2 == 0 or (l == 3):
                tr = rand_seq(rng, len(tr))                       # junk: fails min_read_align_score
            if l % 8 == 2 and r == 1:
                tr = motif * kk + rand_seq(rng, 75 * m)           # the length estimate is 75 copies off: iteration budget
            segs.append(SegmentShim(f"read{l}_{r}", bool(rng.integers(0, 2)), 15000, tr, mutate(rng, fl, 0.01, 0, 0) or "A",
                                    mutate(rng, fr, 0.01, 0, 0) or "A", m))
        loci.append((motif, segs))
    return loci


def run_block_vs_per_call(loci, engine, per_call, rc_params):
    """Block mode (one BlockSession for all loci, then the unchanged loop bound to its look-ups) against per-call mode
    (the same loop calling `per_call` read by read): read dictionaries and log lines must be identical."""
    from strkit_b200.locus_block import BlockSession
    from tests.ref_loop_shim import read_loop

    session = BlockSession(rc_params, engine=engine)
    for motif, segs in loci:
        session.add_locus(motif, [(s.get_est_copy_num(), s.tr_seq_wc, s.flank_left_seq_wc, s.flank_right_seq_wc) for s in segs])
    session.run()
    n_abandoned = n_budget = 0
    for motif, segs in loci:
        want = read_loop(motif, segs, per_call, rc_params)
        got = read_loop(motif, segs, session.get_repeat_count, rc_params)
        assert got == want, motif
        n_abandoned += want[0] is None
        n_budget += any("maximum # iterations" in ln for ln in want[1])
    assert session.misses == 0 and session.hits > 0      # the device replayed exactly the calls the loop makes
    assert n_abandoned >= 1 and n_budget >= 1            # the abort and the budget log line were exercised
    return session


def test_block_session_equals_per_call_loop_host_logic(oracle):
    from strkit_b200 import RepeatCountParams

    p = RepeatCountParams("repalign", 50, 3, 1)

    def per_call(start_count, tr_seq, flank_left_seq, flank_right_seq, motif, rc_params):
        return oracle.get_repeat_count(start_count, tr_seq, flank_left_seq, flank_right_seq, motif, rc_params.max_iters,
                                       rc_params.initial_local_search_range, rc_params.initial_step_size)

    eng = _CheckerEngine(oracle)
    session = run_block_vs_per_call(make_block_loci(), eng, per_call, p)
    assert eng.calls == 1                                 # one device call for the whole block
    # reference windows: warmed the same way; a call that was not collected is a miss (answered per call)
    from strkit_b200 import get_reference_rc_params

    rp = get_reference_rc_params("repalign", 20, 250)
    args = (20, "CAG" * 20, "ACGTTGCATGCATTGACCATGACTGAATCG", "TTGACGATCGGATCGATTAGCTAGCTAAGC", "CAG", 60, 5, rp)
    session.add_reference(*args)
    session.run()
    want = oracle.get_ref_repeat_count(*args[:7], rp.max_iters, rp.initial_local_search_range, rp.initial_step_size)
    assert session.get_ref_repeat_count(*args) == want and session.ref_hits == 1 and session.ref_misses == 0
