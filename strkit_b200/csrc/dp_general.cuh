// dp_general.cuh -- general semi-global DP kernel (int32 lanes, any length, any alphabet).
//
// One CTA of GEN_WARPS warps per alignment family.  The rows of the DP matrix (db = fl + tr + fr, the sequence the
// reference profiles, repeats.py:91-93) are cut into strips: lane t owns R consecutive rows, the
// warp sweeps the columns (the candidate) as a skewed wavefront -- at step s lane t computes
// column s - t + 1 -- and the bottom cell of lane t-1 reaches lane t through __shfl_up_sync.
// Families longer than 32*R rows take several strips, pipelined over the warps of the CTA (see GenSync); the boundary
// row between two strips travels through a ring of scratch rows in global memory (L2-resident).
//
// The candidate fl + motif*n + fr is never materialised (reference builds it with
// f"{fl}{motif * i}{fr}"): columns are generated on the fly from the left flank and the motif
// period.  All candidate sizes of a window share ONE forward sweep: because column |fl| + m*n of
// the sweep against fl + motif*n_hi is the state after fl + motif*n, and the remaining |fr|
// columns of any candidate only depend on db's suffix, score(n) = max_i F[i][|fl|+m*n] + B[i],
// where B is one backward sweep of reverse(fr) against reverse(db).  Max-plus path
// decomposition: exact, not a heuristic.
//
// Rows are FRONT-padded to a multiple of 32*R with copy rows (see dp_pass), so the last real row is
// always the last register of lane 31 and the init row needs no special case.
//
// Linear gaps only: the reference passes open = extend = 5 (repeats.py:33,40), so parasail's
// affine recurrence collapses to H = max(diag + s, max(up, left) - g), evaluated on biased cells
// H' = H + g * (row + column) as H' = max3(diag' + (s + 2g), up', left') (dp_pass).
#pragma once
#include "strk_common.cuh"

#define STRK_NEG_INF (-(1 << 29))

enum PassKind { PASS_DUMP = 0, PASS_COMBINE = 1, PASS_ARGMAX = 2 };

struct PassCfg {
    const unsigned char *s1;   // rows (db), n1 symbols
    const unsigned char *pre;  // column prefix
    const unsigned char *motif;
    int n1, n_pre, m;
    int rev_s1, rev_pre, rev_motif;
    int n_lo, n_hi;       // candidate sizes (COMBINE / ARGMAX)
    int ncols;            // n_pre + m * n_hi  (DUMP: n_pre)
    int s1_beg_free;      // column-0 border is 0
    int s1_last_special;  // backward sweep of a free s1 end: row n1 is not a start node
    int s2_beg_free;      // top border is 0
    int kind;
    int lastrow_term;     // COMBINE with a free s2 end: candidates may stop early on the last row
    int *B;               // [n1 + 2] DUMP writes, COMBINE reads; B[n1 + 1] = best score of a path that
                          // starts inside the suffix columns (free s2 begin), see dp_pass
    int *out;             // COMBINE: [n_hi - n_lo + 1], pre-set to STRK_NEG_INF
    long long *out64;     // ARGMAX: packed (score << 32 | 0x7fffffff - row), pre-set to LLONG_MIN
    int *rows;            // boundary-row scratch: (warps of the CTA + 1) rows of rowlen ints (multi-strip families only)
    int rowlen;
};

// A family is swept by the GEN_WARPS warps of one CTA: warp w takes the strips w, w + GEN_WARPS, ... and the strips
// run as a pipeline -- strip b + 1 follows strip b about 64 columns behind, reading the boundary row strip b leaves
// in the ring slot b % (warps + 1).  A long read (config 4: 12 strips of 6 200 columns) is bound by the latency of its
// own dependency chain, so four strips in flight cut its time almost four-fold.  progress[slot] = b * stride + last
// column written: values only grow over the strips that reuse a slot, so a stale value never satisfies a waiter.
#ifndef GEN_WARPS
#define GEN_WARPS 4
#endif
#define GEN_WARPS_MAX 16  // most warps a CTA may be launched with (512 threads x 128 registers = one SM's file)
#define GEN_STRIP_ROWS (32 * 16)  // rows of one strip (R = 16, strk_pick_rows): a longer family is swept in several
#define GEN_RING_MAX (GEN_WARPS_MAX + 1)  // ring of boundary rows / progress counters: (warps of the CTA) + 1 slots in use
#define GEN_FAST_MMAX 256  // longest motif / prefix (flank) whose column tables a sweep keeps in shared memory; longer
#define GEN_FAST_PMAX 256  // ones take the general loop with a symbol fetch per column
struct GenSync {
    volatile long long progress[GEN_RING_MAX];
    unsigned int q;
};

struct SmemConsts {
    unsigned char lut[256];
    signed char smat[STRK_SMAT_ROWS * STRK_NSYM_];
};

__device__ __forceinline__ int border_col0(const PassCfg &c, int i, int g) {
    // H[i][0] for real row i (i <= 0: pad rows and the corner)
    if (i <= 0) return 0;
    if (c.s1_beg_free) return (c.s1_last_special && i == c.n1) ? -g : 0;
    return -g * i;
}
__device__ __forceinline__ int border_row0(const PassCfg &c, int j, int g) { return c.s2_beg_free ? 0 : -g * j; }

// Scoring tables of the general kernel in shared memory.  Cells are held BIASED: cell (I, j) of the padded matrix
// stores H + g * (I + j), which turns the linear-gap recurrence into  H' = max3(diag' + (s + 2g), up', left')  --
// one add and one three-input max per cell, and a dependency chain of one max per row down a lane's strip.
struct GenSmem {
    unsigned char lut[256];
    short smat2[STRK_SMAT_ROWS * STRK_NSYM_];  // [row symbol or pad][column symbol], score + 2g
    unsigned long long t8[STRK_NSYM_];         // PRMT byte table per column symbol: byte c = score(row class c) + 2g
    unsigned char cls[STRK_SMAT_ROWS + 1];     // row symbol -> PRMT class (A C G T N X other pad), 0x80 = none
    unsigned one;                              // = 1, opaque to the compiler: multiplier of the FMA-pipe adds
    // byte tables of the columns of the sweep in progress, in sweep order: [0, n_pre) the prefix (flank) columns, then
    // the m columns of one motif copy (tC[n_pre + k] = t8[symbol of the k-th column of a copy]).  A lane walks it with
    // one LDS.64 per step and an offset that wraps from the end of the copy back to its start -- no symbol fetch
    // (global load -> code table -> byte table, a chain of three loads) on the critical path of a step.
    unsigned long long tC[2][GEN_FAST_PMAX + GEN_FAST_MMAX];  // [1]: second of two side-by-side sweeps (process_ref_family)
};

__device__ __forceinline__ int gen_add(int a, int b, unsigned one) {  // a + b as IMAD (FMA pipe)
    int r;
    asm("mad.lo.s32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"((int)one), "r"(b));
    return r;
}
__device__ __forceinline__ unsigned gen_prmt(unsigned a, unsigned b, unsigned sel) {
    unsigned r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
    return r;
}

// Steady-state steps of a sweep: every lane is inside the matrix and no lane can reach a candidate column -- for a 6 kb
// expansion that is ~97 % of the steps.  What is left of the general loop's
// bookkeeping: one LDS.64 of the column's byte table with a wrapping offset, the two shuffles, the boundary-row
// store of lane 31 and the running maximum of the last row; everything else (column fetch with its flank / motif /
// reverse cases, activity tests, candidate detection) is compiled out.  TOP / BOT / PM are uniform per strip.
//   TOP: the strip reads the boundary row of the strip above;  BOT: it publishes its own last row;
//   PM:  the running maximum of the last row is needed (last strip, free s2 end).
template <int R, bool TOP, bool BOT, bool PM>
__device__ __forceinline__ void gen_fast_steps(int (&H)[R], const unsigned (&sel)[R], int &prev_up, int &s, const int s_end,
                                               const int lane, const unsigned one, const unsigned long long *tC, const int endb,
                                               const int wrapb, int koff, int topv, const int tinc, int &top_cur, int &top_nxt,
                                               const int *__restrict__ top, int *__restrict__ bot, const int ncols,
                                               volatile long long *prog_in, volatile long long *prog_out,
                                               const long long stride, const int b, int &pmax, const int g) {
    // Whole chunks of 32 steps, entered with s a multiple of 32: the boundary-row refill (TOP) and the progress
    // publication (BOT) happen between chunks, the 32 steps in between are straight-line and convergent (lane 31's
    // boundary-row store is predicated, not branched).
    const char *tbase = (const char *)tC;  // koff: byte offset of this lane's column; endb -> wrapb at the end of a copy
    int gj = g * (s - lane + 1);  // g * (column of this lane)
    const unsigned on31 = lane == 31 ? 1u : 0u;
#pragma unroll 1
    for (; s + 32 <= s_end; s += 32) {
        if (TOP) {
            top_cur = top_nxt;
            if (s + 33 <= ncols) {
                const long long need = (long long)(b - 1) * stride + (s + 64 < ncols ? s + 64 : ncols);
                while (*prog_in < need) __nanosleep(40);
                __threadfence_block();
                if (s + 33 + lane <= ncols) top_nxt = __ldcg(top + s + 33 + lane);
            }
        }
        int *botp = BOT ? bot + (s - 30) : nullptr;  // lane 31 is at column s + k - 30 in step s + k
#pragma unroll 2
        for (int k = 0; k < 32; ++k) {
            int up_in = __shfl_up_sync(0xffffffffu, H[R - 1], 1);
            if (TOP) {
                const int t0 = __shfl_sync(0xffffffffu, top_cur, k);
                up_in = lane == 0 ? t0 : up_in;
            } else {
                up_in = lane == 0 ? topv : up_in;
                topv += tinc;
            }
            const unsigned long long t = *(const unsigned long long *)(tbase + koff);
            koff += 8;
            koff = koff == endb ? wrapb : koff;
            const unsigned tlo = (unsigned)t, thi = (unsigned)(t >> 32);
            int d = prev_up, u = up_in;
            prev_up = up_in;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int left = H[r];
                const int tt = gen_add(d, (int)gen_prmt(tlo, thi, sel[r]), one);
                const int h = max(max(tt, u), left);
                d = left;
                u = h;
                H[r] = h;
            }
            if (BOT)
                asm volatile("{ .reg .pred p; setp.ne.u32 p, %2, 0; @p st.global.u32 [%0], %1; }" ::"l"(botp + k), "r"(H[R - 1]),
                             "r"(on31)
                             : "memory");
            if (PM) {
                pmax = max(pmax, H[R - 1] - gj);
                gj += g;
            }
        }
        if (BOT) {
            if (lane == 31) {  // the row is complete up to column s + 1 (lane 31's column in the chunk's last step)
                __threadfence();
                *prog_out = (long long)b * stride + (s + 1);
            }
            __syncwarp();
        }
    }
}

// One sweep.  LUT = true: every row symbol of the family is A/C/G/T/N/X/other (or pad) and the score of a cell is a
// PRMT byte select from the column's 8-byte table (PRMT + IMAD + VIMNMX3 per cell); LUT = false (IUPAC codes inside
// the read): a shared-memory look-up per cell.
// Pad rows (front padding) are COPY rows: their score entry is 0 (= -2g + 2g), so with up' >= diag' and
// up' >= left' each one repeats the value above it; lane 0 of the first strip injects DP row 0 biased as the last
// pad row (index off), which is what the first real row then reads as its up / diagonal neighbour.
// Block-level opening of a sweep: the previous sweep of the family is complete, the strip pipeline is reset and the
// motif's byte tables (sweep order) are in shared memory.  `slot` = which of the two table slots the sweep uses.
template <bool LUT>
__device__ __forceinline__ bool dp_pass_open(const PassCfg &c, const GenSmem &sc, GenSync &sy, int slot, bool first) {
    if (first) {
        __syncthreads();  // the previous sweep of this family is complete (its B column, its boundary rows)
        if (threadIdx.x < GEN_RING_MAX) sy.progress[threadIdx.x] = -1;
    }
    const bool fast_ok = LUT && c.m <= GEN_FAST_MMAX && c.n_pre <= GEN_FAST_PMAX;
    if (fast_ok) {
        unsigned long long *t = const_cast<GenSmem &>(sc).tC[slot];
        for (int k = threadIdx.x; k < c.n_pre; k += blockDim.x) t[k] = sc.t8[sc.lut[c.pre[c.rev_pre ? c.n_pre - 1 - k : k]]];
        if (c.ncols > c.n_pre)  // (the backward sweep of a read family stops at the end of its prefix)
            for (int k = threadIdx.x; k < c.m; k += blockDim.x)
                t[c.n_pre + k] = sc.t8[sc.lut[c.motif[c.rev_motif ? c.m - 1 - k : k]]];
    }
    return fast_ok;
}

// `warp` = the (virtual) warp index of the caller within the sweep: warp w takes strips w, w + GEN_WARPS, ...
template <int R, bool LUT>
__device__ void dp_pass_body(const PassCfg &c, const GenSmem &sc, GenSync &sy, int g, const int warp, const int slot,
                             const bool fast_ok) {
    const int lane = threadIdx.x & 31;
    const int RB = 32 * R;
    const int NB = c.n1 <= RB ? 1 : (c.n1 + RB - 1) / RB;
    const int off = NB * RB - c.n1;  // number of pad rows in front
    const unsigned one = sc.one;

    if (c.kind == PASS_DUMP && c.ncols == 0) {  // no columns: the last column is the border
        if (warp == 0) {
            for (int i = lane; i <= c.n1; i += 32) c.B[i] = border_col0(c, i, g);
            if (lane == 0) c.B[c.n1 + 1] = border_col0(c, c.n1, g);
        }
        return;
    }
    // candidate column 0 (empty left flank and n = 0): scores come from the border column
    if (warp == 0 && c.kind == PASS_COMBINE && c.n_pre == 0 && c.n_lo == 0) {
        int best = STRK_NEG_INF;
        for (int i = lane; i <= c.n1; i += 32) {
            int b = c.B[c.n1 - i];
            // node (n1, 0) is not an end node: with a free s2 end the path must take one more column
            if (i == c.n1 && c.lastrow_term) b = -g;
            best = max(best, border_col0(c, i, g) + b);
        }
        if (c.s2_beg_free && lane == 0) best = max(best, c.B[c.n1 + 1]);
        atomicMax(&c.out[0], best);
    }

    const long long stride = (long long)c.ncols + 2;
    const int nw = (int)(blockDim.x >> 5), ring = nw + 1;  // (dp_pass_pair: one strip per sweep, nw is not used)
    for (int b = warp; b < NB; b += nw) {
        const int Ibase = b * RB + lane * R;  // padded index of the row above my strip
        int H[R];
        unsigned sel[R];  // LUT: PRMT selector; else: row offset into smat2
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int I = Ibase + r + 1, i = I - off;  // real row 1..n1, <= 0 for pad rows
            int code = STRK_PAD_PEN;
            if (i >= 1) code = sc.lut[c.s1[c.rev_s1 ? c.n1 - i : i - 1]];
            sel[r] = LUT ? ((unsigned)(sc.cls[code] & 7u) | 0x8880u) : (unsigned)(code * STRK_NSYM_);
            H[r] = i >= 1 ? border_col0(c, i, g) + g * I : g * off;
        }
        int prev_up = Ibase - off >= 1 ? border_col0(c, Ibase - off, g) + g * Ibase : g * off;  // row above, column 0
        // (a sweep without columns computes no cell: nothing is published, nothing may be waited for)
        const int *top = b == 0 || c.ncols == 0 ? nullptr : c.rows + (size_t)((b - 1) % ring) * c.rowlen;
        int *bot = b < NB - 1 ? c.rows + (size_t)(b % ring) * c.rowlen : nullptr;
        volatile long long *prog_in = &sy.progress[(b + ring - 1) % ring];
        volatile long long *prog_out = &sy.progress[b % ring];
        // wait until the strip above has published its boundary row up to column `col` (clipped to the last one)
        auto wait_top = [&](int col) {
            const long long need = (long long)(b - 1) * stride + (col < c.ncols ? col : c.ncols);
            while (*prog_in < need) __nanosleep(40);
            __threadfence_block();
        };
        // boundary row of the strip above: fetched 32 columns at a time (one coalesced load per 32 steps, issued 32
        // steps before its first use) and handed to lane 0 by shuffle -- a per-step load by lane 0 would put an L2
        // round trip on every step of a multi-strip read
        int top_cur = 0, top_nxt = 0;
        if (top) {
            wait_top(32);
            if (1 + lane <= c.ncols) top_nxt = __ldcg(top + 1 + lane);
        }
        int pmax = STRK_NEG_INF;  // running max of (last row - g * j): lane 31 of the last strip
        int ncop = 0;
        // the column one step ahead: its symbol (and byte table) is fetched while the current column is computed
        int kk_cur = -1, kk_nxt = -1;
        unsigned long long t_nxt = 0ull;
        int code_nxt = 0;
        // fast_ok: the column tables of the sweep are in shared memory (sc.tC[slot]) and ko walks them
        const char *tbase = (const char *)sc.tC[slot];
        const int endb = (c.n_pre + c.m) * 8, wrapb = c.n_pre * 8;
        int ko = 0;  // byte offset of the next column to fetch
        auto fetch = [&](int jn) {
            if (jn < 1 || jn > c.ncols) return;
            if (jn > c.n_pre) kk_nxt = kk_nxt + 1 == c.m ? 0 : kk_nxt + 1;
            if (LUT && fast_ok) {
                t_nxt = *(const unsigned long long *)(tbase + ko);
                ko += 8;
                ko = ko == endb ? wrapb : ko;
                return;
            }
            if (jn <= c.n_pre)
                code_nxt = sc.lut[c.pre[c.rev_pre ? c.n_pre - jn : jn - 1]];
            else
                code_nxt = sc.lut[c.motif[c.rev_motif ? c.m - 1 - kk_nxt : kk_nxt]];
            if (LUT) t_nxt = sc.t8[code_nxt];
        };
        fetch(1 - lane);
        const int row0_bias = g * off;
        const int nsteps = c.ncols + 31;
        // steady-state range [s_a, s_b): every lane is inside the matrix (s >= 31), lane 0 has not reached the first
        // candidate column (n_pre + m * n_lo, at step n_pre + m * n_lo - 1; the backward sweep: its last column)
        int s_a = 32, s_b = c.kind == PASS_DUMP ? c.ncols - 1 : c.n_pre + c.m * c.n_lo - 1;  // (whole 32-step chunks)
        if (s_b > c.ncols - 1) s_b = c.ncols - 1;
        s_b = s_b < s_a ? s_a : s_a + ((s_b - s_a) & ~31);
        if (!fast_ok || s_b - s_a < 32) s_a = s_b = nsteps;  // not worth it: one general loop
        for (int s = 0; s < nsteps; ++s) {
            if (LUT && s == s_a) {
                const int j0 = s - lane;  // columns before this lane's: j0 <= n_pre -> prefix entry j0, else motif entry
                const int koff = (j0 < c.n_pre ? j0 : c.n_pre + (j0 - c.n_pre) % c.m) * 8;
                const int topv = border_row0(c, s + 1, g) + row0_bias + g * (s + 1);
                const int tinc = c.s2_beg_free ? g : 0;
                const bool pm = b == NB - 1;  // (only read there; cheap enough to keep for every last strip)
#define GEN_FAST(TOPF, BOTF, PMF)                                                                                       \
    gen_fast_steps<R, TOPF, BOTF, PMF>(H, sel, prev_up, s, s_b, lane, one, sc.tC[slot], endb, wrapb, koff, topv, tinc, top_cur, top_nxt, \
                                       top, bot, c.ncols, prog_in, prog_out, stride, b, pmax, g)
                if (top) {
                    if (bot)
                        GEN_FAST(true, true, false);
                    else if (pm)
                        GEN_FAST(true, false, true);
                    else
                        GEN_FAST(true, false, false);
                } else {
                    if (bot)
                        GEN_FAST(false, true, false);
                    else if (pm)
                        GEN_FAST(false, false, true);
                    else
                        GEN_FAST(false, false, false);
                }
#undef GEN_FAST
                // back to the general loop at step s = s_b: restore its one-column-ahead fetch state and the count of
                // motif copies this lane has completed (last computed column: s - lane)
                const int jn = s - lane + 1;  // (1 <= jn: s >= 31; jn may lie past the last column at the end of a sweep)
                kk_nxt = jn > c.n_pre ? (jn - c.n_pre - 1) % c.m : -1;
                ko = (jn <= c.n_pre ? jn - 1 : c.n_pre + kk_nxt) * 8;
                if (jn <= c.ncols) {
                    t_nxt = *(const unsigned long long *)(tbase + ko);
                    ko += 8;
                    ko = ko == endb ? wrapb : ko;
                }
                ncop = s - lane > c.n_pre ? (s - lane - c.n_pre) / c.m : 0;
                if (s >= nsteps) break;
            }
            const int j = s - lane + 1;
            int up_in = __shfl_up_sync(0xffffffffu, H[R - 1], 1);
            const bool active = j >= 1 && j <= c.ncols;
            if (top) {
                if ((s & 31) == 0) {
                    top_cur = top_nxt;
                    if (s + 33 <= c.ncols) {
                        wait_top(s + 64);
                        if (s + 33 + lane <= c.ncols) top_nxt = __ldcg(top + s + 33 + lane);
                    }
                }
                const int t0 = __shfl_sync(0xffffffffu, top_cur, s & 31);  // top[s + 1]: lane 0 is at column s + 1
                if (lane == 0) up_in = t0;
            } else if (lane == 0) {
                up_in = border_row0(c, j, g) + row0_bias + g * j;  // DP row 0, biased as row `off`
            }
            const unsigned long long t_cur = t_nxt;
            const int code_cur = code_nxt;
            kk_cur = kk_nxt;
            fetch(j + 1);
            if (!active) continue;
            int d = prev_up, u = up_in;
            prev_up = up_in;
            if (LUT) {
                const unsigned tlo = (unsigned)t_cur, thi = (unsigned)(t_cur >> 32);
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int left = H[r];
                    const int t = gen_add(d, (int)gen_prmt(tlo, thi, sel[r]), one);
                    const int h = max(max(t, u), left);
                    d = left;
                    u = h;
                    H[r] = h;
                }
            } else {
                const short *srow = sc.smat2 + code_cur;
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int left = H[r];
                    const int h = max(max(d + (int)srow[sel[r]], u), left);
                    d = left;
                    u = h;
                    H[r] = h;
                }
            }
            if (bot && lane == 31) {
                bot[j] = H[R - 1];
                if ((j & 31) == 0 || j == c.ncols) {  // publish: the row is complete up to column j
                    __threadfence();  // the consumer reads the row from L2 (ld.cg): the stores must have got there
                    *prog_out = (long long)b * stride + j;
                }
            }
            pmax = max(pmax, H[R - 1] - g * j);

            // candidate column?
            int n = -1;
            if (c.kind == PASS_DUMP) {
                if (j == c.ncols) n = 0;
            } else if (j == c.n_pre) {
                n = 0;
            } else if (j > c.n_pre && kk_cur == c.m - 1) {
                n = ++ncop;
            }
            if (n < 0) continue;
            const int bias1 = g * (Ibase + 1 + j);  // bias of my first row at this column
            if (c.kind == PASS_DUMP) {
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    int i = Ibase + r + 1 - off;
                    if (i >= 0) c.B[i] = H[r] - bias1 - g * r;
                }
                if (off == 0 && b == 0 && lane == 0) c.B[0] = border_row0(c, j, g);
            } else if (n >= c.n_lo && n <= c.n_hi) {
                const int pmax_unb = pmax - g * (NB * RB);  // meaningful on lane 31 of the last strip
                if (c.kind == PASS_COMBINE) {
                    int best = STRK_NEG_INF;
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        int i = Ibase + r + 1 - off;
                        if (i >= 0) best = max(best, H[r] - bias1 - g * r + c.B[c.n1 - i]);
                    }
                    if (off == 0 && b == 0 && lane == 0) best = max(best, border_row0(c, j, g) + c.B[c.n1]);
                    if (c.lastrow_term && b == NB - 1 && lane == 31) best = max(best, pmax_unb);
                    // free s2 begin: a path may start on the top border to the right of this column
                    if (c.s2_beg_free && b == NB - 1 && lane == 31) best = max(best, c.B[c.n1 + 1]);
                    atomicMax(&c.out[n - c.n_lo], best);
                } else {  // ARGMAX over real rows i >= 1, smallest row on ties (parasail end_query = i - 1)
                    long long best = (long long)0x8000000000000000ull;
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        int i = Ibase + r + 1 - off;
                        if (i >= 1) {
                            long long key = ((long long)(H[r] - bias1 - g * r) << 32) | (unsigned)(0x7fffffff - i);
                            best = key > best ? key : best;
                        }
                    }
                    atomicMax(&c.out64[n - c.n_lo], best);
                }
            }
        }
        // backward sweep: best value anywhere on its last row (= forward row 0, i.e. paths that skip the
        // whole prefix through a free s2 begin), including the border cell
        if (c.kind == PASS_DUMP && b == NB - 1 && lane == 31)
            c.B[c.n1 + 1] = max(pmax - g * (NB * RB), border_col0(c, c.n1, g));
    }
}

template <int R, bool LUT>
__device__ void dp_pass(const PassCfg &c, const GenSmem &sc, GenSync &sy, int g) {
    const bool fast_ok = dp_pass_open<LUT>(c, sc, sy, 0, true);
    __syncthreads();
    dp_pass_body<R, LUT>(c, sc, sy, g, threadIdx.x >> 5, 0, fast_ok);
}

// Two independent single-strip sweeps side by side: warp 0 runs `a`, warp 1 runs `b` (the forward and the reverse
// sg_qe alignment of a reference window).  A one-strip sweep occupies one warp and is bound by the latency of its own
// dependency chain, so the pair takes the time of one.
template <int R, bool LUT>
__device__ void dp_pass_pair(const PassCfg &a, const PassCfg &b, const GenSmem &sc, GenSync &sy, int g) {
    const bool fa = dp_pass_open<LUT>(a, sc, sy, 0, true);
    const bool fb = dp_pass_open<LUT>(b, sc, sy, 1, false);
    __syncthreads();
    const int warp = threadIdx.x >> 5;
    if (warp == 0)
        dp_pass_body<R, LUT>(a, sc, sy, g, 0, 0, fa);
    else if (warp == 1)
        dp_pass_body<R, LUT>(b, sc, sy, g, 0, 1, fb);
}

// true when every symbol of the family's db has a PRMT row class (no IUPAC code inside the read)
__device__ inline bool rows_have_classes(const unsigned char *s1, int n1, const GenSmem &sc) {
    bool ok = true;
    for (int i = threadIdx.x & 31; i < n1; i += 32) ok = ok && !(sc.cls[sc.lut[s1[i]]] & 0x80);
    return __all_sync(0xffffffffu, ok);
}

// ---------------------------------------------------------------------------------------------
// Read family: B = backward sweep of reverse(fr) vs reverse(db); then the forward sweep of
// fl + motif*n_hi vs db combines at every candidate column.  `flags` = STRK_*_FREE end flags.
// ---------------------------------------------------------------------------------------------
template <int R>
__device__ void process_read_family(const FamDesc &f, const unsigned char *arena, const GenSmem &sc, GenSync &sy, int g,
                                    int flags, int *table, int *scratch, int scratch_rowlen, int scratch_b_len) {
    const int n1 = f.n_fl + f.n_tr + f.n_fr;
    const int W = f.n_hi - f.n_lo + 1;
    int *out = table + f.out_off;
    for (int k = threadIdx.x; k < W; k += blockDim.x) out[k] = STRK_NEG_INF;  // (dp_pass opens with a barrier)

    const bool lut_ok = rows_have_classes(arena + f.db_off, n1, sc);
    PassCfg c;
    c.s1 = arena + f.db_off;
    c.n1 = n1;
    c.motif = arena + f.motif_off;
    c.m = f.m;
    c.B = scratch;
    c.rows = scratch + scratch_b_len;
    c.rowlen = scratch_rowlen;
    c.out = out;
    c.out64 = nullptr;
    c.n_lo = f.n_lo;
    c.n_hi = f.n_hi;

    // backward sweep: rows reverse(db), columns reverse(fr); its begin flags are the end flags
    c.pre = arena + f.db_off + f.n_fl + f.n_tr;
    c.n_pre = f.n_fr;
    c.rev_s1 = 1;
    c.rev_pre = 1;
    c.rev_motif = 0;
    c.ncols = f.n_fr;
    c.s1_beg_free = (flags & 2) != 0;
    c.s1_last_special = 1;
    c.s2_beg_free = (flags & 8) != 0;
    c.kind = PASS_DUMP;
    c.lastrow_term = 0;
    if (lut_ok)
        dp_pass<R, true>(c, sc, sy, g);
    else
        dp_pass<R, false>(c, sc, sy, g);

    // forward sweep
    c.pre = arena + f.db_off;
    c.n_pre = f.n_fl;
    c.rev_s1 = 0;
    c.rev_pre = 0;
    c.ncols = f.n_fl + f.m * f.n_hi;
    c.s1_beg_free = (flags & 1) != 0;
    c.s1_last_special = 0;
    c.s2_beg_free = (flags & 4) != 0;
    c.kind = PASS_COMBINE;
    c.lastrow_term = (flags & 8) != 0;
    if (lut_ok)
        dp_pass<R, true>(c, sc, sy, g);
    else
        dp_pass<R, false>(c, sc, sy, g);
}

// ---------------------------------------------------------------------------------------------
// Reference-boundary family (score_ref_boundaries, repeats.py:23-43): two sg_qe sweeps.
//   fwd: columns fl + motif*n           rows db            -> out64[2*k]
//   rev: columns reverse(fr) + reverse(motif)*n   rows reverse(db)   -> out64[2*k + 1]
// ---------------------------------------------------------------------------------------------
template <int R>
__device__ void process_ref_family(const FamDesc &f, const unsigned char *arena, const GenSmem &sc, GenSync &sy, int g,
                                   long long *table, int *scratch, int scratch_rowlen, int scratch_b_len) {
    const int n1 = f.n_fl + f.n_tr + f.n_fr;
    const int W = f.n_hi - f.n_lo + 1;
    long long *out = table + 2 * f.out_off;
    for (int k = threadIdx.x; k < 2 * W; k += blockDim.x) out[k] = (long long)0x8000000000000000ull;

    const bool lut_ok = rows_have_classes(arena + f.db_off, n1, sc);
    PassCfg c;
    c.s1 = arena + f.db_off;
    c.n1 = n1;
    c.motif = arena + f.motif_off;
    c.m = f.m;
    c.B = nullptr;
    c.rows = scratch + scratch_b_len;
    c.rowlen = scratch_rowlen;
    c.out = nullptr;
    c.n_lo = f.n_lo;
    c.n_hi = f.n_hi;
    c.s1_beg_free = 0;  // sg_qe: both begins penalised, end of s1 free
    c.s1_last_special = 0;
    c.s2_beg_free = 0;
    c.kind = PASS_ARGMAX;
    c.lastrow_term = 0;

    c.pre = arena + f.db_off;
    c.n_pre = f.n_fl;
    c.rev_s1 = 0;
    c.rev_pre = 0;
    c.rev_motif = 0;
    c.ncols = f.n_fl + f.m * f.n_hi;
    c.out64 = out;
    PassCfg cr = c;
    cr.pre = arena + f.db_off + f.n_fl + f.n_tr;
    cr.n_pre = f.n_fr;
    cr.rev_s1 = 1;
    cr.rev_pre = 1;
    cr.rev_motif = 1;
    cr.ncols = f.n_fr + f.m * f.n_hi;
    cr.out64 = out + W;
    if (n1 <= 32 * R && c.ncols > 0 && cr.ncols > 0) {  // one strip each: the two sweeps run on two warps at once
        if (lut_ok)
            dp_pass_pair<R, true>(c, cr, sc, sy, g);
        else
            dp_pass_pair<R, false>(c, cr, sc, sy, g);
        return;
    }
    if (lut_ok)
        dp_pass<R, true>(c, sc, sy, g);
    else
        dp_pass<R, false>(c, sc, sy, g);
    if (lut_ok)
        dp_pass<R, true>(cr, sc, sy, g);
    else
        dp_pass<R, false>(cr, sc, sy, g);
}

// Persistent kernel: CTAs (GEN_WARPS warps on one family) pull families from a cost-sorted queue.
template <bool REF>
__global__ void __launch_bounds__(GEN_WARPS_MAX * 32, 1) dp_general_kernel(const FamDesc *__restrict__ fams, const int *__restrict__ order,
                                                         int n_fams, const unsigned char *__restrict__ arena,
                                                         const ScoreConsts *__restrict__ consts, void *table,
                                                         int *scratch, int scratch_rowlen, int scratch_b_len,
                                                         unsigned int *queue,
                                                         const unsigned int *__restrict__ n_fams_dev) {
    if (n_fams_dev) n_fams = (int)*n_fams_dev;  // list length produced on the device (packed-kernel fallbacks)
    __shared__ GenSmem sc;
    __shared__ GenSync sy;
    const int g = consts->gap;
    for (int k = threadIdx.x; k < 256; k += blockDim.x) sc.lut[k] = consts->lut[k];
    for (int k = threadIdx.x; k < STRK_SMAT_ROWS * STRK_NSYM_; k += blockDim.x) sc.smat2[k] = (short)(consts->smat[k] + 2 * g);
    for (int k = threadIdx.x; k < STRK_NSYM_; k += blockDim.x) sc.t8[k] = consts->t8f[k];
    // (a matrix whose biased scores do not fit a positive byte has no byte tables: every family takes the look-up path)
    for (int k = threadIdx.x; k <= STRK_SMAT_ROWS; k += blockDim.x) sc.cls[k] = consts->packed_ok ? consts->cls_of[k] : 0x80;
    if (threadIdx.x == 0) sc.one = consts->one_v[0];
    __syncthreads();
    const int flags = consts->end_flags;
    int *my_scratch = scratch + (size_t)blockIdx.x * ((size_t)scratch_b_len + (size_t)((blockDim.x >> 5) + 1) * scratch_rowlen);

    for (;;) {
        __syncthreads();  // every warp is done with the previous family (and has read sy.q)
        if (threadIdx.x == 0) sy.q = atomicAdd(queue, 1u);
        __syncthreads();
        const unsigned int q = sy.q;
        if (q >= (unsigned)n_fams) break;
        const FamDesc f = fams[order ? order[q] : (int)q];
        const int n1 = f.n_fl + f.n_tr + f.n_fr;
        const int R = strk_pick_rows(n1, (int)(blockDim.x >> 5));
#define STRK_CASE(RR)                                                                                          \
    case RR:                                                                                                   \
        if (REF)                                                                                               \
            process_ref_family<RR>(f, arena, sc, sy, g, (long long *)table, my_scratch, scratch_rowlen,        \
                                   scratch_b_len);                                                             \
        else                                                                                                   \
            process_read_family<RR>(f, arena, sc, sy, g, flags, (int *)table, my_scratch, scratch_rowlen,      \
                                    scratch_b_len);                                                            \
        break;
        switch (R) {
            STRK_CASE(2)
            STRK_CASE(3)
            STRK_CASE(4)
            STRK_CASE(5)
            STRK_CASE(6)
            STRK_CASE(7)
            STRK_CASE(8)
            STRK_CASE(9)
            STRK_CASE(10)
            STRK_CASE(12)
            STRK_CASE(14)
            default:
                STRK_CASE(16)
        }
#undef STRK_CASE
    }
}
