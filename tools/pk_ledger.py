#!/usr/bin/env python
"""Per-read instruction ledger of the packed DP kernel: step loops against everything else, per rows-per-lane class.

    cuobjdump -sass strkit_b200/libstrkit_b200.so > all.sass
    python tools/pk_ledger.py all.sass [--loci 4096] [--seed S] [--ref] [--instr-per-read R=N ...]

Trip counts come from warp_steps(), a copy of the kernel's step-range arithmetic (dp_packed.cuh: the tract split
b0, the window, the flank / motif phases and the capture regions), over the reads of bench.py's config-2 generator
(synth.generate on the CPU; candidate window est +- 6, the read path's first window).  Loop bodies come from the
SASS: leaf loops of a class's kernel that carry the R VIMNMX3.U16x2 of a step are step loops (LDS.64 = motif phase,
stores = captures); the other leaf loops are per-read loops (staging, column tables, profile, combine, reference
reduction), counted with their trip counts; instructions of the read loop outside every leaf loop count once per
read.  That "static" remainder is an estimate: branches inside the read loop are counted as taken.  With
--instr-per-read R=N (warp instructions per read of class R, e.g. from a profiler) the remainder is N minus the step
loops instead.
"""
from __future__ import annotations

import argparse
import collections
import math
import os
import re
import sys

WB = 4       # combine: candidates per batch of loads (dp_packed.cuh)
WBR = 2      # reference-mode epilogue: columns per batch of loads
WINDOW = 6   # read path's first window: est +- 6
PAIR_RMAX = 8  # classes up to this are swept two reads per warp, 16 lanes x 2R rows (api.cu pk_lanes_for_class)


def _cdiv(a: int, b: int) -> int:
    """C integer division (truncates toward zero), as the kernel computes b0."""
    q = abs(a) // abs(b)
    return q if (a >= 0) == (b > 0) else -q


def warp_steps(reads, L: int = 32, ref_mode: bool = False) -> dict:
    """Trip counts of one warp of the packed kernel.  reads: one read (L = 32) or one or two (L = 16, the two units of
    the warp), each (n_fl, n_tr, n_fr, m, n_lo, n_hi).  Copies dp_packed.cuh: the tract split and window, the step
    ranges (warp-wide max / min), then the steps of each region the kernel runs a separate loop for."""
    SK = L - 1
    units = []
    for n_fl, n_tr, n_fr, m, n_lo, n_hi in reads:
        b0 = _cdiv(m * n_hi + n_fl - n_fr + m, 2 * m)
        b0 = 0 if b0 < 0 else min(b0, n_lo)
        if ref_mode:
            b0 = 0
        a_lo, a_hi = n_lo - b0, n_hi - b0
        nW = a_hi - a_lo + 1
        nWB = nW if ref_mode else 1
        if ref_mode:
            b0 = n_hi
        colsF, colsB = n_fl + m * a_hi, n_fr + m * b0
        units.append(dict(n1=n_fl + n_tr + n_fr, m=m, b0=b0, a_lo=a_lo, a_hi=a_hi, nW=nW, nWB=nWB, colsF=colsF,
                          colsB=colsB, ncols=max(colsF, colsB), first_cand=n_fl + m * a_lo,
                          first_candB=colsB - m * (nWB - 1), flank=max(n_fl, n_fr)))
    Lmax = max(u["flank"] for u in units)
    nsteps = max(u["ncols"] + SK for u in units)
    s_star = min(Lmax + SK, nsteps)
    fc_begin = min(u["first_cand"] - 1 for u in units)
    bc_begin = min(u["first_candB"] - 1 for u in units)
    bc_end = max(u["colsB"] + SK for u in units)
    e0 = min(s_star, SK)
    ramp_caps = fc_begin < e0 or bc_begin < e0
    steps = collections.Counter()
    for s in range(nsteps):
        fc, bc = s >= fc_begin, bc_begin <= s < bc_end
        if s < e0:
            steps["flank_caps" if ramp_caps else "flank"] += 1
        elif s < s_star:
            steps["flank_caps" if fc or bc else "flank"] += 1
        else:
            steps["motif" + ("_fc" if fc else "") + ("_bc" if bc else "")] += 1
    return dict(units=units, Lmax=Lmax, nsteps=nsteps, s_star=s_star, fc_begin=fc_begin, bc_begin=bc_begin,
                bc_end=bc_end, ramp=e0, ramp_caps=ramp_caps, steps=dict(steps),
                colt_entries=Lmax + 2 * SK + 1)


# ---------------------------------------------------------------- SASS side
def find_loops(ins, text):
    """(first, last) instruction index of every loop closed by a backward branch."""
    idx = {a: i for i, (a, _) in enumerate(ins)}
    out = []
    for i, t in enumerate(text):
        m = re.search(r"BRA(?:\.\w+)*\s+(?:!?U?P\d+,\s*)?0x([0-9a-f]+)", t)
        if m:
            tgt = int(m.group(1), 16)
            if tgt <= ins[i][0] and tgt in idx:
                out.append((idx[tgt], i))
    return sorted(set(out))


def classify(ops: collections.Counter, R: int) -> str:
    if ops["VIMNMX3.U16x2"] == R and ops["SHFL.UP"] >= 1:
        stores = sum(v for k, v in ops.items() if k.startswith("STG"))
        if ops["LDS.64"]:
            return "motif" if not stores else f"motif_st{stores}"
        if ops["PRMT"] == R and ops["IMAD"] <= R + 2:
            return "flank" if not stores else "flank_caps"
        return "flank_other"
    if ops["CREDUX.MAX"] and ops["VIADDMNMX.U16x2"]:
        return "combine_batch" if ops["VIADDMNMX.U16x2"] > R else "combine_one"
    if ops["CREDUX.MAX"]:
        return "ref_batch" if ops["CREDUX.MAX"] > 1 else "ref_column"
    if ops["LDG.E.U8.CONSTANT"] and ops["ISETP.LT.U32.AND"]:
        return "stage_motif"
    if ops["LDG.E.U8.CONSTANT"] and ops["LDS.U8"]:
        return "stage_read"
    if ops["STS.U8"] and not ops["LDG.E.U8.CONSTANT"]:
        return "stage_pad"
    if ops["PRMT"] and (ops["STS"] or ops["STS.64"]):
        return "profile"
    if ops["LDS.S8"]:
        return "profile_general"
    if ops["CS2R"] and ops["LDS.U8"]:
        return "colt"
    return "other"


def kernel_ledger(lines, R: int, L: int):
    ins_full = []
    pat = f"dp_packed_kernelILi{R}ELi{L}E"
    start = next(i for i, l in enumerate(lines) if "Function :" in l and pat in l)
    end = next((i for i in range(start + 1, len(lines)) if "Function :" in lines[i]), len(lines))
    rx = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(.*?);")
    for l in lines[start:end]:
        m = rx.search(l)
        if m:
            ins_full.append((int(m.group(1), 16), m.group(2).strip()))
    text = [t for _, t in ins_full]
    ops_of = [re.sub(r"^@!?U?P\w+\s+", "", t).split()[0] for t in text]
    lps = find_loops(ins_full, text)
    outer = max(lps, key=lambda p: p[1] - p[0])
    # leaf loops of the read loop (the out-of-line warp-collective fallbacks after it close "loops" of their own)
    leaves = [p for p in lps if not any(q != p and p[0] <= q[0] and q[1] <= p[1] for q in lps)
              and outer[0] <= p[0] and p[1] <= outer[1]]
    body = {}
    for a, b in leaves:
        ops = collections.Counter(ops_of[a:b + 1])
        body.setdefault(classify(ops, R), []).append(b - a + 1)
    in_leaf = sum(b - a + 1 for a, b in leaves)
    return dict(body=body, straight=(outer[1] - outer[0] + 1) - in_leaf, n_ins=len(ins_full))


def step_body(body, variant: str, R: int) -> float:
    """SASS length of the loop a step region runs in."""
    if variant.startswith("flank"):
        lst = body.get(variant) or body.get("flank_other") or [0]
        return min(lst)
    if variant == "motif":
        return min(body.get("motif", [0]))
    caps = sorted((int(k.split("_st")[1]), min(v)) for k, v in body.items() if k.startswith("motif_st"))
    if not caps:
        return 0
    if variant == "motif_fc_bc":
        return caps[-1][1]
    return caps[0][1]


def per_read_loops(body, ws, L: int, R: int, ref_mode: bool) -> float:
    """Instructions of the per-read leaf loops of one warp iteration (trip counts from warp_steps)."""
    u = ws["units"]
    n1 = max(x["n1"] for x in u)
    m = max(x["m"] for x in u)
    nW = max(x["nW"] for x in u)
    tot = 0.0
    for role, lens in body.items():
        ln = min(lens)
        if role == "stage_read":
            tot += ln * math.ceil(n1 / L / 4)
        elif role == "stage_motif":
            tot += ln * math.ceil(m / L / 4)
        elif role == "stage_pad":
            tot += ln * math.ceil((L * R - n1) / L / 8)
        elif role == "colt":
            tot += ln * math.ceil(ws["colt_entries"] / L)
        elif role == "profile":
            prmt_cols = 1 if ln < 4 * R else (2 if ln < 8 * R else 4)
            tot += ln * math.ceil(m / prmt_cols)
        elif role == "combine_batch" and not ref_mode:
            one = "combine_one" in body
            tot += ln * (nW // WB if one else math.ceil(nW / WB))
        elif role == "combine_one" and not ref_mode:
            tot += ln * (nW % WB)
        elif role == "ref_batch" and ref_mode:  # both directions, WBR = 2 columns per batch
            tot += sum(lens) * (nW // WBR) / len(lens) * 2
        elif role == "ref_column" and ref_mode:  # one column per trip: the remainder of the batches, or every column
            tot += sum(lens) * (nW % WBR if "ref_batch" in body else nW) / len(lens) * 2
    return tot


def workload(n_loci: int, seed: int):
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from strkit_b200 import synth

    b = synth.generate(synth.CONFIGS[2], n_loci, seed=seed).to_host()
    loc = (b.read_begin[1:] - b.read_begin[:-1])
    locus_of = [i for i, n in enumerate(loc.tolist()) for _ in range(n)]
    out = []
    for r in range(b.n_reads):
        fl, tr, fr = (int(x) for x in b.lens[r])
        m = int(b.motif_len[locus_of[r]])
        est = int(b.est_cn[r])
        out.append((fl, tr, fr, m, max(est - WINDOW, 0), est + WINDOW))
    return out


def pk_class(fl, tr, fr, m):
    R = max(2, (fl + tr + fr + 1 + 31) // 32)
    if R > 16 or fl < 1 or fr < 1 or fl > 160 or fr > 160 or m * R > 128 or m <= 0:
        return 0
    return R


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("sass")
    ap.add_argument("--loci", type=int, default=4096)
    ap.add_argument("--seed", type=int, default=20261018 + 2000)
    ap.add_argument("--ref", action="store_true", help="reference mode (window est +- 6 as well)")
    ap.add_argument("--instr-per-read", nargs="*", default=[], help="R=N: measured warp instructions per read")
    args = ap.parse_args()
    measured = {int(k): float(v) for k, v in (x.split("=") for x in args.instr_per_read)}
    lines = open(args.sass).read().splitlines()
    reads = workload(args.loci, args.seed)
    by_class = collections.defaultdict(list)
    for rd in reads:
        R = pk_class(rd[0], rd[1], rd[2], rd[3])
        if R:
            by_class[R].append(rd)
    mode = "reference" if args.ref else "reads"
    print(f"# {mode} mode, {len(reads)} reads of {args.loci} config-2 loci; warp instructions per read")
    print(f"{'R':>2s} {'kernel':>12s} {'reads':>6s} {'steps':>6s} {'step-loop instr':>16s}  {'remainder':>9s} {'share':>6s}  by variant")
    for R in sorted(by_class):
        L = 16 if R <= PAIR_RMAX else 32
        KR = 2 * R if L == 16 else R
        try:
            led = kernel_ledger(lines, KR, L)
        except StopIteration:
            print(f"{R:2d} kernel <{KR}, {L}> not in the dump")
            continue
        rs = by_class[R]
        per = 32 // L
        tot_steps, tot_loop, tot_rem = 0.0, 0.0, 0.0
        var = collections.Counter()
        for i in range(0, len(rs), per):
            ws = warp_steps(rs[i:i + per], L, args.ref)
            for v, n in ws["steps"].items():
                c = n * step_body(led["body"], v, KR)
                var[v] += c
                tot_loop += c
                tot_steps += n
            tot_rem += led["straight"] + per_read_loops(led["body"], ws, L, KR, args.ref)
        n = len(rs)
        loop_pr, rem_pr = tot_loop / n, tot_rem / n
        src = "static"
        if R in measured:
            rem_pr, src = measured[R] - loop_pr, "measured"
        share = rem_pr / (rem_pr + loop_pr)
        vs = ", ".join(f"{k} {v / n:.0f}" for k, v in sorted(var.items()))
        print(f"{R:2d} {f'<{KR},{L}>':>12s} {n:6d} {tot_steps / n:6.0f} {loop_pr:16.0f}  {rem_pr:9.0f} {share:6.1%}  "
              f"{vs}  ({src}; straight-line {led['straight']})")


if __name__ == "__main__":
    main()
