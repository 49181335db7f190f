"""CPU tests of tools/pk_ledger.warp_steps: the packed kernel's trip-count arithmetic (tract split, window, flank /
motif phases, capture regions) against reads worked out by hand from dp_packed.cuh."""
import importlib.util
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ledger():
    spec = importlib.util.spec_from_file_location("pk_ledger", os.path.join(ROOT, "tools", "pk_ledger.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_read_mode_one_read_per_warp():
    # fl 70, tract 150, fr 70, motif 3, est 50 -> window [44, 56]
    # b0 = (3 * 56 + 70 - 70 + 3) / 6 = 28; a = 16..28 (13 candidates); forward / backward columns 70 + 3 * 28 = 154
    # steps 154 + 31 = 185; motif phase from 70 + 31 = 101; captures from 70 + 3 * 16 - 1 = 117 (forward) and
    # 154 - 1 = 153 (the final backward column) until 185
    ws = _ledger().warp_steps([(70, 150, 70, 3, 44, 56)], L=32)
    u = ws["units"][0]
    assert (u["b0"], u["a_lo"], u["a_hi"], u["nW"], u["nWB"]) == (28, 16, 28, 13, 1)
    assert (u["colsF"], u["colsB"], u["ncols"]) == (154, 154, 154)
    assert (ws["Lmax"], ws["nsteps"], ws["s_star"]) == (70, 185, 101)
    assert (ws["fc_begin"], ws["bc_begin"], ws["bc_end"]) == (117, 153, 185)
    assert (ws["ramp"], ws["ramp_caps"]) == (31, False)
    assert ws["steps"] == {"flank": 101, "motif": 16, "motif_fc": 36, "motif_fc_bc": 32}
    assert ws["colt_entries"] == 70 + 62 + 1


def test_reference_mode_captures_every_size_on_both_halves():
    # reference mode: b0 = 0 for the forward half, both halves sweep fl / fr + 3 * 56 = 238 columns and capture the
    # 13 sizes from column 70 + 3 * 44 = 202 on
    ws = _ledger().warp_steps([(70, 150, 70, 3, 44, 56)], L=32, ref_mode=True)
    u = ws["units"][0]
    assert (u["b0"], u["a_lo"], u["a_hi"], u["nW"], u["nWB"]) == (56, 44, 56, 13, 13)
    assert (u["colsF"], u["colsB"], u["first_cand"], u["first_candB"]) == (238, 238, 202, 202)
    assert (ws["nsteps"], ws["fc_begin"], ws["bc_begin"], ws["bc_end"]) == (269, 201, 201, 269)
    assert ws["steps"] == {"flank": 101, "motif": 100, "motif_fc_bc": 68}


def test_tract_split_clamps_and_truncates_like_c():
    # numerator 2 * 10 + 1 - 150 + 2 = -127 < 0: b0 = 0 (C division truncates, then the clamp at 0)
    u = _ledger().warp_steps([(1, 20, 150, 2, 0, 10)], L=32)["units"][0]
    assert (u["b0"], u["a_lo"], u["a_hi"]) == (0, 0, 10)
    # b0 above n_lo: clamped to n_lo
    u = _ledger().warp_steps([(150, 40, 1, 4, 2, 8)], L=32)["units"][0]
    assert (u["b0"], u["a_lo"], u["a_hi"], u["nW"]) == (2, 0, 6, 7)
    assert _ledger()._cdiv(-127, 4) == -31 and _ledger()._cdiv(127, 4) == 31


def test_two_reads_per_warp_share_the_step_ranges():
    # 16 lanes per read (skew 15): the warp runs the union -- longest flank, last step, first capture of either read
    a = (40, 60, 30, 2, 24, 36)   # b0 = (72 + 40 - 30 + 2) / 4 = 21; a = 3..15; cols 40 + 30 = 70 / 30 + 42 = 72
    b = (20, 90, 50, 3, 24, 36)   # b0 = (108 + 20 - 50 + 3) / 6 = 13; a = 11..23; cols 20 + 69 = 89 / 50 + 39 = 89
    ws = _ledger().warp_steps([a, b], L=16)
    ua, ub = ws["units"]
    assert (ua["b0"], ua["a_lo"], ua["colsF"], ua["colsB"]) == (21, 3, 70, 72)
    assert (ub["b0"], ub["a_lo"], ub["colsF"], ub["colsB"]) == (13, 11, 89, 89)
    assert ws["Lmax"] == 50 and ws["nsteps"] == 89 + 15 and ws["s_star"] == 65
    assert ws["fc_begin"] == min(40 + 2 * 3, 20 + 3 * 11) - 1 == 45
    assert ws["bc_begin"] == 71 and ws["bc_end"] == 89 + 15
    # ramp 0..14 and flank steps up to 44 without captures, 45..64 flank steps with them (the first forward candidate
    # of read a comes before the motif phase), then 65..70 forward only, 71..103 both
    assert ws["steps"] == {"flank": 45, "flank_caps": 20, "motif_fc": 6, "motif_fc_bc": 33}
