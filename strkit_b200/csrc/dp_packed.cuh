// dp_packed.cuh -- packed u16x2 DPX kernel for the bulk of the reads (db < 512 bases).
//
// Same strip wavefront as dp_general.cuh (lane t owns R consecutive rows of db, columns swept with a
// one-column skew per lane, bottom cell handed down with __shfl_up_sync), but every 32-bit lane word
// carries TWO sweeps of the same read at once:
//     low  half: forward sweep   rows db            columns fl + motif*a          (a <= a_hi)
//     high half: backward sweep  rows reverse(db)   columns reverse(fr) + reverse(motif)*b0
// and score(n = a + b0) = max_i F[i][|fl| + m*a] + B[n1 - i][|fr| + m*b0]: the candidate is split in the
// MIDDLE of its repeat tract, so both halves sweep about half of the candidate and one pass of
// (|cand| / 2 + 31) steps scores the whole window of sizes.  Exact max-plus path decomposition.
//
// Cell update in 2 integer instructions.  With H' = H + g*(row + col) the linear-gap recurrence
//     H = max(diag + s, max(up, left) - g)      becomes      H' = max3(diag' + (s + 2g), up', left')
// i.e. one add (an IMAD, so that it issues on the FMA pipe) and one VIMNMX3.U16x2 written in place; every H' is
// >= 0, so unsigned 16-bit lanes never underflow and a plain 32-bit add cannot carry between the halves.
//
// Substitution scores without a per-cell table walk:
//   * flank phase (columns still inside fl / fr): PRMT as an 8-entry byte LUT.  The 8-byte table comes
//     from the column symbol (one shared-memory load per step), the selector from the row symbol (fixed
//     register), the upper byte of each half is produced by PRMT's sign-replicate mode.  Per cell pair:
//     PRMT + IMAD + VIMNMX3 for a read whose rows are all A/C/G/T (FLANK0), one more IMAD when rows hold X / N
//     wildcards (FLANK1: their score rides along as a per-row addend), two PRMT otherwise (FLANK2).
//   * motif phase (both halves inside the periodic tract): the pair of column symbols repeats with
//     period m, so a packed query profile is built once per read in shared memory (stored as row pairs) and
//     the step costs LDS.64 / 2 + IMAD.IADD + VIMNMX3 per cell pair.  The candidate is never materialised.
//
// The step loops are branch-free.  Lanes that have not started yet (column <= 0) run on an all-zero score
// table, which leaves their border column untouched (the biased borders are non-decreasing down the rows);
// lanes that are past the last column compute values nobody reads.  Candidate columns (and the final column
// of the backward half) are captured with predicated stores into a per-warp scratch that mostly stays in
// L2; the combine pass reads them back (one candidate per lane for the closing arithmetic).
//
// Rows are front-padded to 32*R (> n1, so there is always at least one pad row, which doubles as DP row 0);
// row n1 is therefore always the last register of lane 31.  Pad rows score zero and so copy the row above them;
// lane 0 injects DP row 0 above its first register (see "borders" in the kernel).
//
// Reads this kernel cannot take (IUPAC codes inside the read, value range beyond u16, empty flank) are
// appended to a fallback list that the general int32 kernel processes afterwards -- still on the GPU.
//
// Reference mode (ref_mode != 0): the same sweeps serve score_ref_boundaries (repeats.py:23-43).  The low halves
// hold the forward sg_qe alignment of a reference window, the high halves the reverse one, both over the whole
// prefix chain and both captured at every size of the window; instead of combining the halves, the epilogue
// reduces each captured column to (best score, smallest row attaining it) = parasail's (score, end_query).
#pragma once
#include "dp_general.cuh"
#include "strk_common.cuh"

#define PK_FLANK_MAX 160  // longest flank the packed kernel stages (reference default flank_size = 70)
#define PK_WINDOW_MAX 128  // widest window (candidate sizes per read) a batch pass gives to the packed kernel
#ifndef PK_WARPS
#define PK_WARPS 4  // warps per CTA, one read per warp
#endif
#ifndef PK_WARPS_PAIRED
#define PK_WARPS_PAIRED 4  // warps per CTA when a warp holds two reads (2-warp CTAs were measured no faster)
#endif
__host__ __device__ constexpr int pk_warps(int L) { return L == 16 ? PK_WARPS_PAIRED : PK_WARPS; }
#ifndef PK_PROF_IMAD
#define PK_PROF_IMAD 0
#endif
#ifndef PK_ONE_VREG
#define PK_ONE_VREG 0
#endif
#ifndef PK_MIN_CTAS  // occupancy the register allocation is held to (shared memory allows about as many)
#define PK_MIN_CTAS(R) ((R) <= 10 ? 5 : ((R) <= 18 ? 4 : 3))
#endif

// Measurement build only (-DPK_PHASE_TIMERS=1, off by default): clock64() phase timers of the per-read code.
// pk_phase_clk[ref_mode][L == 16][R][phase] sums SM cycles over the warps of every launch since the last reset:
// phase 0 = prologue (queue pop, eligibility, staging, tables, profile, borders, step ranges), 1 = step loops,
// 2 = epilogue (combine or reference-mode reduction), 3 = warp iterations that ran the step loops.  Each warp
// accumulates in registers and adds its totals once, when it leaves the work queue.  tools/pk_phase_timers.py reads it.
#ifndef PK_PHASE_TIMERS
#define PK_PHASE_TIMERS 0
#endif
#if PK_PHASE_TIMERS
__device__ unsigned long long pk_phase_clk[2][2][17][4];
#endif

struct PackedDims {
    int colt_entries;  // uint4 entries of the per-column table  (>= max flank + 64)
    int prof_words;    // u32 words of the packed profile        (>= m_max * R * 32)
    int w_max;         // candidate sizes per read
};

// A read is swept by a UNIT of L lanes: L = 32 (one read per warp) or L = 16 (two reads per warp, side by side: half
// the wavefront skew and half the per-step overhead per read, for reads short enough that 16 * R rows hold them).
__host__ __device__ inline int pk_quads(int R) { return (R + 1 + 3) / 4; }  // H[0..R) + the prefix-max word
// Packed profile of the motif phase: rows in pairs, prof[((k * RH + r / 2) * L + lane) * 2 + (r & 1)], so that a
// step fetches its R scores with RH = ceil(R / 2) conflict-free LDS.64 instead of R LDS.32.
__host__ __device__ inline int pk_prof_rows(int R) { return (R + 1) / 2 * 2; }
__host__ __device__ inline int pk_prof_words(int R, int m, int L = 32) { return m * pk_prof_rows(R) * L; }
__host__ __device__ inline size_t pk_scratch_words_per_unit(int R, int w_max, int L = 32) {
    return (size_t)(w_max + 1) * pk_quads(R) * L * 4;
}
// per-unit shared memory: [colT uint4 x colt_entries][prof u32 x prof_words][row symbols + motif bytes]
// row symbols per register row, forward and backward (pad code on pad rows), then the motif
__host__ __device__ inline size_t pk_code_bytes(int R, int L = 32) { return (size_t)(2 * L * R + 128 + 15) / 16 * 16; }
__host__ __device__ inline size_t pk_smem16_per_unit(int R, const PackedDims &d, int L = 32) {
    return (size_t)d.colt_entries + ((size_t)d.prof_words * 4 + 15) / 16 + pk_code_bytes(R, L) / 16;
}
__host__ __device__ inline size_t pk_smem_bytes(int R, const PackedDims &d, int L = 32) {
    return pk_smem16_per_unit(R, d, L) * 16 * pk_warps(L) * (32 / L);
}

// Raw PRMT (generic mode).  NOT __byte_perm: that intrinsic masks the selector with 0x7777, which costs an
// extra LOP and drops bit 3 of each nibble -- the sign-replicate bit used here to produce the zero bytes.
__device__ __forceinline__ unsigned pk_prmt(unsigned a, unsigned b, unsigned sel) {
    unsigned r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
    return r;
}

// a + b on the FMA pipe: IMAD with a multiplier the compiler cannot see through (`one` comes from the constants
// block).  The ALU pipe (PRMT, VIMNMX3; 0.5 warp-instructions per clock per scheduler) bounds the flank-phase step
// loops, so their adds are taken off it.  Variants measured in place (DESIGN.md 5.1): multiplier in a vector
// register (PK_ONE_VREG=1) -2 %, IMAD instead of the compiler's IMAD.IADD in the motif phase (PK_PROF_IMAD=1) +0.4 %.
__device__ __forceinline__ unsigned pk_add(unsigned a, unsigned b, unsigned one) {
    unsigned r;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(one), "r"(b));
    return r;
}

// H = max3(t, u, H) with the destination tied to the H register (keeps ptxas from renaming it and moving it back)
__device__ __forceinline__ void pk_max3_inplace(unsigned &h, unsigned t, unsigned u) {
    asm("{.reg .b32 t1; \n\t"
        "max.u16x2 t1, %1, %2; \n\t"
        "max.u16x2 %0, t1, %0;}\n\t"
        : "+r"(h) : "r"(t), "r"(u));
}

// Per-lane state of one read in flight.  Everything is indexed with compile-time constants after unrolling,
// so the arrays live in registers.
template <int R>
struct PkState {
    unsigned H[R];     // DP cells of my R rows at the current column: forward (low) | backward (high) half
    unsigned selA[R];  // PRMT selector (two-table path: forward half; one-table path: both halves)
    unsigned selB[R];  // two-table path: PRMT selector of the backward half; one-table path: packed addend
    unsigned prev_up, topv, pm;
    int poff;       // word offset of the current profile column (motif phase)
    int cand_step;  // step at which this lane reaches the next forward candidate column
    unsigned foff;  // next forward capture slot: uint4 index into the warp's scratch (lane offset applied)
    int cand_stepB;  // the same for the backward half (read mode: one column; reference mode: one per size)
    unsigned boff;
    unsigned long long pol;  // L2 cache policy of the capture stores (PK_SCRATCH_POLICY bit 1; unused otherwise)
};

// One column of the wavefront -> scratch: H[0..R) then the prefix-max word, word w of the column at
// dst[(w / 4) * L].{x,y,z,w}.  Full quads go out as predicated 128-bit stores; the tail (R % 4 cells and the
// prefix maximum) as 64- / 32-bit pieces, so that no register has to be copied into an aligned quad first.
// Capture scratch and L2.  A read's captured columns (~20 KB) are written once, read back once by the combine a few
// microseconds later and then dead; without a hint every one of those lines is eventually written back to HBM
// (measured: 1.15 GB of DRAM writes per launch of the R = 10 class against ~35 MB of algorithmic bytes).
// PK_SCRATCH_POLICY bit 0: after the combine, the lines of the read are DISCARDED (discard.global.L2: their contents
// are declared dead, so a dirty line is dropped instead of written back); bit 1: the capture stores carry an
// L2::evict_last policy so the lines outlive the streaming arena traffic until then.
#ifndef PK_SCRATCH_POLICY
#define PK_SCRATCH_POLICY 0
#endif
__device__ __forceinline__ unsigned long long pk_l2_policy() {
    unsigned long long pol = 0ull;
#if PK_SCRATCH_POLICY & 2
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
#endif
    return pol;
}
__device__ __forceinline__ void pk_discard_line(const void *p) {
#if PK_SCRATCH_POLICY & 1
    asm volatile("discard.global.L2 [%0], 128;" ::"l"(p) : "memory");
#endif
}
__device__ __forceinline__ void pk_st4(unsigned *p, unsigned a, unsigned b, unsigned c, unsigned d, unsigned on,
                                       unsigned long long pol) {
    (void)pol;
#if PK_SCRATCH_POLICY & 2
    asm volatile("{ .reg .pred p; setp.ne.u32 p, %5, 0; @p st.global.L2::cache_hint.v4.u32 [%0], {%1, %2, %3, %4}, %6; }" ::"l"(p),
                 "r"(a), "r"(b), "r"(c), "r"(d), "r"(on), "l"(pol)
                 : "memory");
#else
    asm volatile("{ .reg .pred p; setp.ne.u32 p, %5, 0; @p st.global.v4.u32 [%0], {%1, %2, %3, %4}; }" ::"l"(p), "r"(a),
                 "r"(b), "r"(c), "r"(d), "r"(on)
                 : "memory");
#endif
}
__device__ __forceinline__ void pk_st2(unsigned *p, unsigned a, unsigned b, unsigned on) {
    asm volatile("{ .reg .pred p; setp.ne.u32 p, %3, 0; @p st.global.v2.u32 [%0], {%1, %2}; }" ::"l"(p), "r"(a), "r"(b), "r"(on)
                 : "memory");
}
__device__ __forceinline__ void pk_st1(unsigned *p, unsigned a, unsigned on) {
    asm volatile("{ .reg .pred p; setp.ne.u32 p, %2, 0; @p st.global.u32 [%0], %1; }" ::"l"(p), "r"(a), "r"(on) : "memory");
}

template <int R, int L>
__device__ __forceinline__ void pk_capture(const PkState<R> &st, uint4 *__restrict__ dst, const unsigned on) {
    constexpr int QF = R / 4, REM = R % 4;  // full quads, cells in the partial one
#pragma unroll
    for (int q = 0; q < QF; ++q)
        pk_st4((unsigned *)(dst + q * L), st.H[4 * q], st.H[4 * q + 1], st.H[4 * q + 2], st.H[4 * q + 3], on, st.pol);
    unsigned *tail = (unsigned *)(dst + QF * L);
    if (REM == 1) {
        pk_st2(tail, st.H[R - 1], st.pm, on);
    } else if (REM == 2) {
        pk_st2(tail, st.H[R - 2], st.H[R - 1], on);
        pk_st1(tail + 2, st.pm, on);
    } else if (REM == 3) {
        pk_st2(tail, st.H[R - 3], st.H[R - 2], on);
        pk_st2(tail + 2, st.H[R - 1], st.pm, on);
    } else {
        pk_st1(tail, st.pm, on);
    }
}

// FLANK1R = one-table path during the ramp-up steps: lanes that have not reached column 1 yet must see a
// zero score, so their addend is masked off
// FLANK0 = one-table path of a read whose rows are all A/C/G/T (or pad): no addend at all, PRMT + IMAD + VIMNMX3
enum { PK_CORE_FLANK2 = 0, PK_CORE_FLANK1 = 1, PK_CORE_PROF = 2, PK_CORE_FLANK1R = 3, PK_CORE_FLANK0 = 4 };

// Steps [s, s_end) of the wavefront; lane t of a unit (`lane` here is the lane WITHIN the unit) computes column
// s - t + 1 in step s.  CORE selects the score
// source, FC / BC switch the predicated captures of forward candidate columns / the final backward column on.
template <int R, int L, int CORE, bool FC, bool BC>
__device__ __forceinline__ void pk_run(PkState<R> &st, int &s, const int s_end, const bool lane0, const int lane,
                                       const unsigned one, const unsigned tinc, const unsigned ginc, const uint4 *__restrict__ ctp,
                                       const unsigned *__restrict__ prof_lane, const int pstride, const int pwrap,
                                       const int m, const int last_cand_step, const int last_cand_stepB,
                                       uint4 *__restrict__ scr) {
    constexpr int QN = (R + 1 + 3) / 4;
#pragma unroll 1
    for (; s < s_end; ++s) {
        unsigned up_in = __shfl_up_sync(0xffffffffu, st.H[R - 1], 1, L);
        st.topv += tinc;
        up_in = lane0 ? st.topv : up_in;
        unsigned d = st.prev_up, u = up_in;
        st.prev_up = up_in;
        if (CORE == PK_CORE_PROF) {
            const uint2 *pp = (const uint2 *)prof_lane + st.poff;  // this lane's row pairs of the current column
            unsigned sc[(R + 1) / 2 * 2];
#pragma unroll
            for (int q = 0; q < (R + 1) / 2; ++q) {
                const uint2 v = pp[q * L];
                sc[2 * q] = v.x;
                sc[2 * q + 1] = v.y;
            }
            unsigned t[R];
#if PK_PROF_IMAD
            t[0] = pk_add(d, sc[0], one);
#pragma unroll
            for (int r = 1; r < R; ++r) t[r] = pk_add(st.H[r - 1], sc[r], one);
#else
            t[0] = d + sc[0];
#pragma unroll
            for (int r = 1; r < R; ++r) t[r] = st.H[r - 1] + sc[r];
#endif
#pragma unroll
            for (int r = 0; r < R; ++r) {
                pk_max3_inplace(st.H[r], t[r], u);
                u = st.H[r];
            }
            st.poff = st.poff + pstride == pwrap ? 0 : st.poff + pstride;
        } else {
            const uint4 ct = ctp[s];  // = colT[column + 31]
            const unsigned started = s >= lane ? one : 0u;
            unsigned t[R];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const unsigned dd = r == 0 ? d : st.H[r == 0 ? 0 : r - 1];
                if (CORE == PK_CORE_FLANK0)
                    t[r] = pk_add(dd, pk_prmt(ct.x, ct.z, st.selA[r]), one);
                else if (CORE == PK_CORE_FLANK1)
                    t[r] = pk_add(pk_add(dd, pk_prmt(ct.x, ct.z, st.selA[r]), one), st.selB[r], one);
                else if (CORE == PK_CORE_FLANK1R)  // addend * (0 | 1): masked on the FMA pipe as well
                    t[r] = pk_add(st.selB[r], pk_add(dd, pk_prmt(ct.x, ct.z, st.selA[r]), one), started);
                else
                    t[r] = pk_add(pk_add(dd, pk_prmt(ct.x, ct.y, st.selA[r]), one), pk_prmt(ct.z, ct.w, st.selB[r]), one);
            }
#pragma unroll
            for (int r = 0; r < R; ++r) {
                pk_max3_inplace(st.H[r], t[r], u);
                u = st.H[r];
            }
        }
        st.pm = __viaddmax_u16x2(st.pm, ginc, st.H[R - 1]);
        if (FC) {  // predicated, not branched: some lane captures in almost every step of the candidate region
            const bool hit = s == st.cand_step;
            pk_capture<R, L>(st, scr + st.foff, hit ? 1u : 0u);
            const int nxt = st.cand_step + m;
            st.foff += hit ? QN * L : 0;
            st.cand_step = hit ? (nxt > last_cand_step ? 0x7fffffff : nxt) : st.cand_step;
        }
        if (BC) {
            const bool hit = s == st.cand_stepB;
            pk_capture<R, L>(st, scr + st.boff, hit ? 1u : 0u);
            const int nxt = st.cand_stepB + m;
            st.boff += hit ? QN * L : 0;
            st.cand_stepB = hit ? (nxt > last_cand_stepB ? 0x7fffffff : nxt) : st.cand_stepB;
        }
    }
}

// max over my rows of forward + paired backward value for one captured candidate column (low halves only)
template <int R, int QN>
__device__ __forceinline__ unsigned pk_cand_max(const uint4 (&c)[QN], const unsigned (&Bv)[R]) {
    unsigned acc = 0u;
#pragma unroll
    for (int q = 0; q < QN; ++q) {
        if (4 * q + 0 < R) acc = __viaddmax_u16x2(c[q].x, Bv[(4 * q + 0) % R], acc);
        if (4 * q + 1 < R) acc = __viaddmax_u16x2(c[q].y, Bv[(4 * q + 1) % R], acc);
        if (4 * q + 2 < R) acc = __viaddmax_u16x2(c[q].z, Bv[(4 * q + 2) % R], acc);
        if (4 * q + 3 < R) acc = __viaddmax_u16x2(c[q].w, Bv[(4 * q + 3) % R], acc);
    }
    return acc & 0xffffu;
}

template <int R, int L>
__global__ void __launch_bounds__(pk_warps(L) * 32, PK_MIN_CTAS(R) * PK_WARPS / pk_warps(L))
dp_packed_kernel(const FamDesc *__restrict__ fams, const int *__restrict__ list, int n_list,
                 const unsigned char *__restrict__ arena, const ScoreConsts *__restrict__ consts,
                 int *__restrict__ table, PackedDims dims, uint4 *__restrict__ scratch,
                 int *__restrict__ fallback_list, unsigned int *__restrict__ fallback_count, int ref_mode,
                 unsigned int *__restrict__ work_counter) {
    static_assert(R >= 2 && (L == 32 || L == 16), "rows per lane / lanes per read out of range");
    constexpr int HALVES = 32 / L;  // reads side by side in one warp
    constexpr int SK = L - 1;       // wavefront skew: lane t of a unit is t columns behind lane 0
    constexpr int N = L * R;
    constexpr int QN = (R + 1 + 3) / 4;
    constexpr int RH = (R + 1) / 2;  // row pairs of the packed profile
    constexpr int WB = 4;   // combine: candidate columns per batch of loads (hides the L2 round trip)
    constexpr int WBR = 2;  // reference mode: columns per batch (with 4, ptxas laid out some classes' step loops worse)
    extern __shared__ uint4 smem_raw[];
    __shared__ SmemConsts sc;
    __shared__ unsigned long long t8f[STRK_NSYM_], t8b[STRK_NSYM_];
    __shared__ unsigned rowinfo[STRK_SMAT_ROWS + 1];
    for (int k = threadIdx.x; k < 256; k += blockDim.x) sc.lut[k] = consts->lut[k];
    for (int k = threadIdx.x; k < STRK_SMAT_ROWS * STRK_NSYM_; k += blockDim.x) sc.smat[k] = consts->smat[k];
    for (int k = threadIdx.x; k < STRK_NSYM_; k += blockDim.x) {
        t8f[k] = consts->t8f[k];
        t8b[k] = consts->t8b[k];
    }
    for (int k = threadIdx.x; k <= STRK_SMAT_ROWS; k += blockDim.x) rowinfo[k] = consts->rowinfo[k];
    __syncthreads();

    const int wlane = threadIdx.x & 31;
    const int lane = wlane & (L - 1);  // lane within the unit: everything below is written per unit
    const int half = wlane / L;
    const unsigned hmask = L == 32 ? 0xffffffffu : (0xffffu << (16 * half));  // the lanes of my unit
    const int warp = threadIdx.x >> 5;
    const int unit = warp * HALVES + half;
    const int unit_global = (blockIdx.x * pk_warps(L) + warp) * HALVES + half;
    const int total_units = gridDim.x * pk_warps(L) * HALVES;
    const int g = consts->gap;
    // reference mode (score_ref_boundaries, repeats.py:23-43): the two halves of a lane word are the two sg_qe
    // alignments of a locus -- every begin penalised, nothing combined; `table` then holds 64-bit (score, end_query) keys
    const int flags = ref_mode ? 0 : consts->end_flags;
    const bool one_table_ok = consts->one_table_ok != 0;
#if PK_ONE_VREG
    const unsigned one = consts->one_v[wlane];  // per-lane load: stays in a vector register
#else
    const unsigned one = consts->one_v[0];  // uniform load
#endif
    const bool s1_beg = flags & 1, s1_end = flags & 2, s2_beg = flags & 4, s2_end = flags & 8;
    const bool lane0 = lane == 0;
    // predicate true on every lane of MY unit (the two units of a warp hold different reads)
    auto all_unit = [&](bool pred) -> bool { return (__ballot_sync(0xffffffffu, pred) & hmask) == hmask; };

    uint4 *colT = smem_raw + (size_t)unit * pk_smem16_per_unit(R, dims, L);  // entry [j + SK], columns -SK .. Lmax + SK
    unsigned *prof = (unsigned *)(colT + dims.colt_entries);
    // symbol codes by REGISTER row (row I of the padded strip, 0-based): rowF[I] = db[I - off], rowB[I] = db[N - 1 - I]
    // (the backward sweep's row), pad code on the pad rows; each lane reads its R consecutive bytes of both
    unsigned char *rowF = (unsigned char *)(prof + (dims.prof_words + 3) / 4 * 4);
    unsigned char *rowB = rowF + N;
    unsigned char *mcodes = rowB + N;
    uint4 *scr = scratch + (size_t)unit_global * (size_t)(dims.w_max + 1) * QN * L;
    const unsigned tinc = (s2_beg ? (unsigned)g : 0u) | ((s2_end ? (unsigned)g : 0u) << 16);
    const unsigned ginc = (unsigned)g | ((unsigned)g << 16);
    const int g2 = 2 * g;

    // Work items come from a queue (one atomic per warp and read, nothing next to a 100-microsecond sweep): a launch
    // that shares the SMs with another context's kernels (the streamed path), or whose CTAs do not all start together,
    // no longer ends on the slowest statically assigned slice.  Both units of a warp take consecutive items.
#if PK_PHASE_TIMERS
    unsigned long long clk_acc[4] = {0ull, 0ull, 0ull, 0ull}, clk_t = clock64();
#define PK_CLK(P)                                      \
    do {                                               \
        const unsigned long long t_ = clock64();       \
        clk_acc[P] += t_ - clk_t;                      \
        clk_t = t_;                                    \
    } while (0)
#else
#define PK_CLK(P) \
    do {          \
    } while (0)
#endif
    // The next item is popped one read ahead while the queue is far from empty (the atomic's latency then hides behind
    // a read); near the end it is popped after the read, so that no warp holds an item while others run out of work.
    unsigned int next = 0u;
    auto pop = [&] {
        if (wlane == 0) next = atomicAdd(work_counter, (unsigned int)HALVES);
    };
    pop();
    bool ahead = false;
    for (;; ahead ? (void)0 : pop()) {
        const unsigned int base = __shfl_sync(0xffffffffu, next, 0);
        if (base >= (unsigned int)n_list) break;
        ahead = base + 2u * (unsigned int)total_units < (unsigned int)n_list;
        if (ahead) pop();
        // a unit without a read of its own in the last round re-runs the last read of the list and stores nothing
        const int fam_idx_raw = (int)base + half;
        const bool have = fam_idx_raw < n_list;
        if (!__any_sync(0xffffffffu, have)) break;
        const int fam_id = list[have ? fam_idx_raw : n_list - 1];
        const FamDesc f = fams[fam_id];
        const int n1 = f.n_fl + f.n_tr + f.n_fr;
        const int off = N - n1;
        const int m = f.m;
        const unsigned char *db = arena + f.db_off;
        const unsigned char *motif = arena + f.motif_off;

        // read mode: split of the tract, b0 copies go to the backward half, candidate n = a + b0.
        // reference mode: both halves sweep the whole prefix chain and are captured at every size of the window.
        int b0 = (m * f.n_hi + f.n_fl - f.n_fr + m) / (2 * m);
        b0 = b0 < 0 ? 0 : (b0 > f.n_lo ? f.n_lo : b0);
        if (ref_mode) b0 = 0;
        const int a_lo = f.n_lo - b0, a_hi = f.n_hi - b0;
        const int nW = a_hi - a_lo + 1;
        const int nWB = ref_mode ? nW : 1;  // captured columns of the backward half
        if (ref_mode) b0 = f.n_hi;          // columns of the backward half: reverse(fr) + reverse(motif) * n_hi
        const int colsF = f.n_fl + m * a_hi, colsB = f.n_fr + m * b0;
        const int ncols = colsF > colsB ? colsF : colsB;
        // the flank phase ends for both units of the warp together: the longer flank of the two reads counts
        const int Lmax = __reduce_max_sync(0xffffffffu, f.n_fl > f.n_fr ? f.n_fl : f.n_fr);

        // ---- eligibility (per warp: with two units, both reads go to the general kernel if either is odd)
        bool ok = off >= 1 && f.n_fl >= 1 && f.n_fr >= 1 && Lmax <= PK_FLANK_MAX && Lmax + 2 * SK + 2 <= dims.colt_entries &&
                  pk_prof_words(R, m, L) <= dims.prof_words && m <= 128 && nW + nWB <= dims.w_max + 1 &&
                  (g * (N + ncols + 40) + 2 * N + 1024) < (ref_mode ? 32000 : 65535);
        ok = __all_sync(0xffffffffu, ok);
        if (!ok) {
            if (lane0 && have) fallback_list[atomicAdd(fallback_count, 1u)] = fam_id;
            continue;
        }
        __syncwarp();  // the previous read's shared-memory readers are done

        // ---- stage the encoded read and motif in shared memory (one coalesced pass over the arena bytes)
        bool motif_acgt = true;
        for (int d = lane; d < n1; d += L) {
            const unsigned char c = sc.lut[db[d]];
            rowF[d + off] = c;
            rowB[N - 1 - d] = c;
        }
        for (int I = lane; I < off; I += L) rowF[I] = rowB[I] = (unsigned char)STRK_PAD_PEN;
        for (int k = lane; k < m; k += L) {
            const unsigned char c = sc.lut[motif[k]];
            mcodes[k] = c;
            motif_acgt = motif_acgt && c < 4;
        }
        motif_acgt = all_unit(motif_acgt);
        __syncwarp();

        // x % m for 0 <= x < 4096 without a division: x - m * ((x * inv) >> 20), inv = ceil(2^20 / m)
        const unsigned inv_m = (1048576u + (unsigned)m - 1u) / (unsigned)m;
        auto mod_m = [&](int x) -> int { return x - (int)(((unsigned)x * inv_m) >> 20) * m; };

        // ---- per-column PRMT tables for the flank phase: columns -SK .. Lmax + SK (zero tables for j <= 0).
        // One-table path: possible when every column symbol of the phase is A/C/G/T (then the score of a
        // non-ACGT row symbol does not depend on the column and rides along as an addend).
        bool acgt = true;
        for (int e = lane; e <= Lmax + 2 * SK; e += L) {
            const int j = e - SK;
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            if (j >= 1) {
                const int sf = j <= f.n_fl ? rowF[off + j - 1] : mcodes[mod_m(j - f.n_fl - 1)];
                const int sb = j <= f.n_fr ? rowF[N - j] : mcodes[m - 1 - mod_m(j - f.n_fr - 1)];
                acgt = acgt && sf < 4 && sb < 4;
                const unsigned long long a = t8f[sf], b = t8b[sb];
                v = make_uint4((unsigned)a, (unsigned)(a >> 32), (unsigned)b, (unsigned)(b >> 32));
            }
            colT[e] = v;
        }
        const bool cols_acgt = all_unit(acgt);

        // ---- row symbols -> PRMT selectors (one-table format first: the profile build uses it too).  One look-up
        // per row and direction: rowinfo[code] holds the selector nibbles, the class, the addend and the flags.
        PkState<R> st;
        const unsigned char *myF = rowF + lane * R, *myB = rowB + lane * R;
        unsigned flags_or = 0u;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const unsigned wf = rowinfo[myF[r]], wb = rowinfo[myB[r]];
            flags_or |= wf | wb;
            // bytes 0-3 of the pair {forward table, backward table} = forward classes, 4-7 = backward classes;
            // selector nibble 8 = sign-replicate of byte 0 = 0x00
            st.selA[r] = (wf & 0xfu) | ((wb & 0xf0u) << 4) | 0x8080u;
            st.selB[r] = ((wf >> 16) & 0xffu) | (wb & 0xff0000u);
        }
        const bool rows_ok = !(flags_or & 0x800u);
        const bool rows_plain = !(flags_or & 0x1000u);  // A/C/G/T or pad only: no row carries an addend
        if (!__all_sync(0xffffffffu, rows_ok)) {  // IUPAC code inside a read of this warp
            if (lane0 && have) fallback_list[atomicAdd(fallback_count, 1u)] = fam_id;
            continue;
        }
        // one table per step is enough when the column-independent addend is exact: either every flank-phase
        // column is A/C/G/T (a non-ACGT row then scores the same in every column), or no row carries an addend
        // (rows all A/C/G/T or pad) -- in which case the step is PRMT + IMAD + VIMNMX3 per cell pair (FLANK0).
        // The step loops are shared by the units of a warp, so the weaker of their cores is taken.
        const bool no_addend = __all_sync(0xffffffffu, rows_plain);
        const bool plain_unit = all_unit(rows_plain);  // evaluated by every lane (it votes across the warp)
        const bool one_table = __all_sync(0xffffffffu, (one_table_ok && cols_acgt) || plain_unit);
        // ---- packed profile for the motif phase (row pairs, see pk_prof_rows), column j = Lmax + 1 + k (mod m)
        // motif positions of column k stepped instead of reduced mod m per column; one base pointer per lane
        {
            int jf = mod_m(Lmax - f.n_fl), jb = m - 1 - mod_m(Lmax - f.n_fr);
            unsigned *pc = prof + 2 * lane;
            if (one_table_ok && motif_acgt) {
                for (int k = 0; k < m; ++k, pc += 2 * RH * L) {
                    const unsigned tf = (unsigned)t8f[mcodes[jf]], tb = (unsigned)t8b[mcodes[jb]];
#pragma unroll
                    for (int r = 0; r < R; ++r) pc[(r >> 1) * 2 * L + (r & 1)] = pk_prmt(tf, tb, st.selA[r]) + st.selB[r];
                    jf = jf + 1 == m ? 0 : jf + 1;
                    jb = jb == 0 ? m - 1 : jb - 1;
                }
            } else {
                for (int k = 0; k < m; ++k, pc += 2 * RH * L) {
                    const int sf = mcodes[jf], sb = mcodes[jb];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const int vf = sc.smat[myF[r] * STRK_NSYM_ + sf] + g2;
                        const int vb = sc.smat[myB[r] * STRK_NSYM_ + sb] + g2;
                        pc[(r >> 1) * 2 * L + (r & 1)] = (unsigned)vf | ((unsigned)vb << 16);
                    }
                    jf = jf + 1 == m ? 0 : jf + 1;
                    jb = jb == 0 ? m - 1 : jb - 1;
                }
            }
        }
        if (!one_table) {
#pragma unroll
            for (int r = 0; r < R; ++r) {
                st.selA[r] = ((rowinfo[myF[r]] >> 8) & 7u) | 0x8880u;
                st.selB[r] = (((rowinfo[myB[r]] >> 8) & 7u) << 8) | 0x8088u;
            }
        }

        // ---- borders (biased by g * (row + col)).  Pad rows are COPY rows: their score byte is zero, so with
        // up' >= diag' and up' >= left' (biased values never decrease along a row or down a column) each one
        // repeats the value above it; lane 0 injects, as the row above its first register, DP row 0 with the bias
        // of the LAST pad row (index off), which is therefore what every pad row holds and what the first real row
        // reads as its up / diagonal neighbour.  No addend, whatever the begin / end mode.
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int I = lane * R + r + 1, i = I - off;
            int vf = g * off, vb = g * off;  // pad rows: DP row 0 at column 0, biased as row `off`
            if (i >= 1) {
                vf = (s1_beg ? 0 : -g * i) + g * I;
                vb = (s1_end ? (i == n1 ? -g : 0) : -g * i) + g * I;
            }
            st.H[r] = (unsigned)vf | ((unsigned)vb << 16);
        }
        {
            const int I = lane * R, i = I - off;
            int vf = g * off, vb = g * off;
            if (i >= 1) {
                vf = (s1_beg ? 0 : -g * i) + g * I;
                vb = (s1_end ? 0 : -g * i) + g * I;  // i < n1 here
            }
            st.prev_up = (unsigned)vf | ((unsigned)vb << 16);
        }
        st.topv = (unsigned)(g * off) | ((unsigned)(g * off) << 16);  // DP row 0 at column 0 (then + tinc per column)
        st.pm = 0u;    // biased prefix maxima of the last row, both halves (meaningful on the last lane of the unit)
        st.poff = 0;
        st.foff = (unsigned)lane;
        st.boff = (unsigned)(nW * (QN * L) + lane);
        st.pol = pk_l2_policy();

        // step ranges, common to the units of the warp (their union).  Lane t is at column c during step c + t - 1.
        const int first_cand = f.n_fl + m * a_lo;
        const int first_candB = colsB - m * (nWB - 1);
        const int nsteps = __reduce_max_sync(0xffffffffu, ncols + SK);
        const int s_star = Lmax + SK < nsteps ? Lmax + SK : nsteps;              // first motif-phase step
        const int fc_begin = __reduce_min_sync(0xffffffffu, first_cand - 1);    // forward captures: [fc_begin, nsteps)
        const int bc_begin = __reduce_min_sync(0xffffffffu, first_candB - 1);   // backward captures: [bc_begin, bc_end)
        const int bc_end = __reduce_max_sync(0xffffffffu, colsB + SK);
        st.cand_step = first_cand + lane - 1;
        st.cand_stepB = first_candB + lane - 1;
        const int last_cand_step = colsF + lane - 1;
        const int last_cand_stepB = colsB + lane - 1;
        const uint4 *ctp = colT + (SK + 1) - lane;  // ctp[s] = table of the column this lane computes in step s
        const unsigned *prof_lane = prof + 2 * lane;
        const int pstride = RH * L, pwrap = m * RH * L;  // in row pairs (uint2)
        __syncwarp();

#define PK_RUN(CORE, FC, BC, END)                                                                          \
    pk_run<R, L, CORE, FC, BC>(st, s, END, lane0, lane, one, tinc, ginc, ctp, prof_lane, pstride, pwrap, m,     \
                               last_cand_step, last_cand_stepB, scr)

        PK_CLK(0);
        int s = 0;
        // ---- flank phase (PRMT look-ups).  Steps 0..SK-1 are the ramp-up of the unit's last lane, after which
        // the prefix maximum of the last row starts from scratch.
        {
            // part 0: ramp-up steps (captures compiled in only if one can fire this early)
            const int e0 = s_star < SK ? s_star : SK;
            const bool ramp_caps = fc_begin < e0 || bc_begin < e0;
            if (no_addend) {
                if (ramp_caps)
                    PK_RUN(PK_CORE_FLANK0, true, true, e0);
                else
                    PK_RUN(PK_CORE_FLANK0, false, false, e0);
            } else if (one_table) {
                if (ramp_caps)
                    PK_RUN(PK_CORE_FLANK1R, true, true, e0);
                else
                    PK_RUN(PK_CORE_FLANK1R, false, false, e0);
            } else {
                if (ramp_caps)
                    PK_RUN(PK_CORE_FLANK2, true, true, e0);
                else
                    PK_RUN(PK_CORE_FLANK2, false, false, e0);
            }
            st.pm = 0u;
            // part 1: cut where the capture switches change, like the motif phase
            while (s < s_star) {
                const bool fc = s >= fc_begin, bc = s >= bc_begin && s < bc_end;
                int e = s_star;
                if (fc_begin > s && fc_begin < e) e = fc_begin;
                if (bc_begin > s && bc_begin < e) e = bc_begin;
                if (bc_end > s && bc_end < e) e = bc_end;
                if (no_addend) {
                    if (fc || bc)
                        PK_RUN(PK_CORE_FLANK0, true, true, e);
                    else
                        PK_RUN(PK_CORE_FLANK0, false, false, e);
                } else if (one_table) {
                    if (fc || bc)
                        PK_RUN(PK_CORE_FLANK1, true, true, e);
                    else
                        PK_RUN(PK_CORE_FLANK1, false, false, e);
                } else {
                    if (fc || bc)
                        PK_RUN(PK_CORE_FLANK2, true, true, e);
                    else
                        PK_RUN(PK_CORE_FLANK2, false, false, e);
                }
            }
        }
        // ---- motif phase (packed profile from shared memory), cut where the capture switches change
        if (s < nsteps) {
            st.poff = mod_m(s - lane - Lmax) * pstride;  // column s - lane + 1 >= Lmax + 1 on every lane here
            while (s < nsteps) {
                const bool fc = s >= fc_begin, bc = s >= bc_begin && s < bc_end;
                int e = nsteps;
                if (fc_begin > s && fc_begin < e) e = fc_begin;
                if (bc_begin > s && bc_begin < e) e = bc_begin;
                if (bc_end > s && bc_end < e) e = bc_end;
                if (fc) {
                    if (bc)
                        PK_RUN(PK_CORE_PROF, true, true, e);
                    else
                        PK_RUN(PK_CORE_PROF, true, false, e);
                } else {
                    if (bc)
                        PK_RUN(PK_CORE_PROF, false, true, e);
                    else
                        PK_RUN(PK_CORE_PROF, false, false, e);
                }
            }
        }
#undef PK_RUN

        __syncwarp();
        PK_CLK(1);
#if PK_PHASE_TIMERS
        clk_acc[3] += 1ull;
#endif
        // From here on the two units of a warp may run different trip counts (window sizes): every warp-level
        // primitive below names only the lanes of the unit (hmask).
        if (ref_mode) {
            // ---- reference mode: per size, the best cell of the captured column and the smallest row attaining it
            // (parasail end_query), for the forward (low halves, slots 0..nW) and the reverse alignment (high halves,
            // slots nW..2nW).  Key = (score + 32768) << 16 | (0xffff - row): one REDUX per column and direction.
            // score + 32768 = h + (32768 - g * I) - g * p: the row term is a per-read constant, the column term is
            // uniform, and PRMT puts the low 16 bits of the sum above the row code.  Pad rows take selector 0 on a
            // zero byte: key 0, the value the maximum starts from, so they never win.
            long long *out64 = (long long *)table + 2 * f.out_off;
            unsigned rc[R], rk[R], rsel[R];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int I = lane * R + r + 1, i = I - off;
                rc[r] = (unsigned)(32768 - g * I);
                rk[r] = i >= 1 ? (unsigned)(0xffff - i) : 0u;
                rsel[r] = i >= 1 ? 0x5410u : 0u;  // bytes {rk.0, rk.1, x.0, x.1}
            }
            const uint4 *col = scr + lane;  // this lane's quads of captured column 0
            for (int dir = 0; dir < 2; ++dir) {
                if (dir) {  // high halves: the same sum, 16 bits up (no carry comes out of the low half: its addend is 0)
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        rc[r] <<= 16;
                        rsel[r] = rsel[r] ? 0x7610u : 0u;  // bytes {rk.0, rk.1, x.2, x.3}
                    }
                }
                const int p0 = (dir ? f.n_fr : f.n_fl) + m * f.n_lo;
                auto column = [&](const uint4(&c)[QN], int w) {
                    const unsigned gp = (unsigned)(-g * (p0 + m * w)), np = dir ? gp << 16 : gp;
                    unsigned key = 0u;
#pragma unroll
                    for (int q = 0; q < QN; ++q) {
                        const unsigned wv[4] = {c[q].x, c[q].y, c[q].z, c[q].w};
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const int r = 4 * q + j;
                            if (r < R) key = max(key, pk_prmt(rk[r], wv[j] + rc[r] + np, rsel[r]));
                        }
                    }
                    key = __reduce_max_sync(hmask, key);
                    if (lane0 && have) {
                        const int score = (int)(key >> 16) - 32768, row = 0xffff - (int)(key & 0xffffu);
                        out64[dir * nW + w] = ((long long)score << 32) | (long long)(unsigned)(0x7fffffff - row);
                    }
                };
                // WBR columns per batch of loads, so that their L2 round trips overlap
                int w = 0;
                for (; w + WBR <= nW; w += WBR, col += WBR * QN * L) {
                    uint4 q4[WBR][QN];
#pragma unroll
                    for (int b = 0; b < WBR; ++b)
#pragma unroll
                        for (int q = 0; q < QN; ++q) q4[b][q] = col[(b * QN + q) * L];
#pragma unroll
                    for (int b = 0; b < WBR; ++b) column(q4[b], w + b);
                }
#pragma unroll 1
                for (; w < nW; ++w, col += QN * L) {
                    uint4 q1[QN];
#pragma unroll
                    for (int q = 0; q < QN; ++q) q1[q] = col[q * L];
                    column(q1, w);
                }
            }
            __syncwarp();
            for (int ln = lane; ln < 2 * nW * QN * L / 8; ln += L) pk_discard_line(scr + ln * 8);  // 128-byte lines
            __syncwarp();
            PK_CLK(2);
            continue;
        }
        // ---- combine: score(n) for every candidate of the window
        const unsigned *scw = (const unsigned *)scr;
        const unsigned bbase = (unsigned)nW * (QN * L * 4);  // word offset of the backward slot
        unsigned Bv[R];  // backward value paired with each forward row (low half), 0 for pad rows
        {
            // forward row If = lane * R + r + 1 pairs with backward row Ib = N + off - If: consecutive, descending,
            // so its (lane, register) position is stepped instead of divided out per row
            int ib1 = N + off - (lane * R + 1) - 1;  // Ib - 1 for r = 0
            int lb = ib1 / R, rb = ib1 - lb * R;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                unsigned v = 0u;
                if (lane * R + r + 1 >= off) v = scw[bbase + (unsigned)(((rb >> 2) * L + lb) * 4 + (rb & 3))] >> 16;
                Bv[r] = v;
                if (--rb < 0) rb = R - 1, --lb;
            }
        }
        const int bextra = (int)(scw[bbase + (unsigned)(((R >> 2) * L + (L - 1)) * 4 + (R & 3))] >> 16);
        constexpr int CW = QN * L;  // uint4 per captured column
        for (int g0 = 0; g0 < nW; g0 += L) {  // L candidates at a time: lane w keeps the reduced value of g0 + w
            const int gn = nW - g0 < L ? nW - g0 : L;
            const uint4 *col = scr + (size_t)g0 * CW + lane;  // loads at compile-time offsets from one pointer
            unsigned my_v = 0u;
            int k = 0;
            // whole batches without a per-candidate exit, then the remainder one candidate at a time
            for (; k + WB <= gn; k += WB, col += WB * CW) {
                uint4 q4[WB][QN];
#pragma unroll
                for (int b = 0; b < WB; ++b)
#pragma unroll
                    for (int q = 0; q < QN; ++q) q4[b][q] = col[b * CW + q * L];
                const int lk = lane - k;
#pragma unroll
                for (int b = 0; b < WB; ++b) {
                    const unsigned v = __reduce_max_sync(hmask, pk_cand_max<R, QN>(q4[b], Bv));
                    my_v = lk == b ? v : my_v;
                }
            }
#pragma unroll 1
            for (; k < gn; ++k, col += CW) {
                uint4 q1[QN];
#pragma unroll
                for (int q = 0; q < QN; ++q) q1[q] = col[q * L];
                const unsigned v = __reduce_max_sync(hmask, pk_cand_max<R, QN>(q1, Bv));
                my_v = lane == k ? v : my_v;
            }
            if (lane < gn && have) {  // un-bias and close the free-end cases: one candidate per lane
                const int w = g0 + lane;
                const int p = f.n_fl + m * (a_lo + w);
                int best = (int)my_v - g * (N + off + p + colsB);
                if (s2_end) {  // prefix maximum of the last row (forward half), word R of the unit's last lane
                    const unsigned flast = scw[(unsigned)(((w * QN + (R >> 2)) * L + (L - 1)) * 4 + (R & 3))] & 0xffffu;
                    best = max(best, (int)flast - g * (N + p));
                }
                if (s2_beg) {
                    const int border = s1_end ? -g : -g * n1;  // backward cell (n1, 0)
                    best = max(best, max(bextra - g * (N + colsB), border));
                }
                table[f.out_off + w] = best;
            }
        }
        __syncwarp();
        // the captured columns of this read are dead: drop their lines from L2 instead of writing them back
        for (int ln = lane; ln < (nW + 1) * QN * L / 8; ln += L) pk_discard_line(scr + ln * 8);
        __syncwarp();
        PK_CLK(2);
    }
#if PK_PHASE_TIMERS
    if (wlane == 0) {
        unsigned long long *acc = pk_phase_clk[ref_mode ? 1 : 0][L == 16 ? 1 : 0][R];
        for (int k = 0; k < 4; ++k) atomicAdd(acc + k, clk_acc[k]);
    }
#endif
#undef PK_CLK
}
