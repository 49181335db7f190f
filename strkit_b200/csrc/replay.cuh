// replay.cuh -- exact replay of the reference's hill-climb over precomputed score tables.
//
// The DP kernels score a whole window of candidate sizes in parallel; the reference instead walks
// sizes serially (strkit_rust_ext.get_repeat_count, called at repeats.py:58-68; the in-tree
// statement of the same search is repeats.py:100-156) and its answer depends on the start size,
// the visitation order, the iteration budget and the tie-breaks -- it is NOT an arg-max.  climb()
// runs that search verbatim with every "score this size" replaced by a table look-up, so the parallel
// sweep returns bit-identical (n, score, n_explored).  A look-up outside the table window is reported
// as a miss; the host widens the window and runs the locus again.  What a window of the search scores
// is a visitor: climb_single (read path, one score per size) and climb_ref (the boundary search of
// get_ref_repeat_count, a forward and a reverse score per size).
//
// Also replayed here, once for both replay kernels: the per-locus read loop of call_locus.py:1079,1129-1161
// (start guess with the carried offset fraction; float64, round-half-even like CPython's round()).  The
// kernels differ only in where a read's table row comes from.
#pragma once
#include "strk_common.cuh"

#define STRK_MAX_WINDOW 4100  // widest table row the replay can track (bitmap of visited sizes)
#define STRK_SEEN_WORDS ((STRK_MAX_WINDOW + 31) / 32)

struct ClimbResult {
    int best_n, best_score, n_explored;
    int status;  // 0 ok, 1 window miss, 2 nothing scored
    double sum_n;  // sum of the sizes scored (for reference-equivalent cell counts)
    int lo_touched, hi_touched;  // extent of the sizes looked up
};

struct SeenSet {
    unsigned int w[STRK_SEEN_WORDS];
    int lo, hi;
    __host__ __device__ void reset(int lo_, int hi_) {
        lo = lo_;
        hi = hi_;
        int nw = (hi_ - lo_ + 32) / 32;
        for (int k = 0; k < nw; ++k) w[k] = 0u;
    }
    __host__ __device__ bool inside(int n) const { return n >= lo && n <= hi; }
    // sizes outside the window can never have been scored
    __host__ __device__ bool has(int n) const {
        if (!inside(n)) return false;
        int k = n - lo;
        return (w[k >> 5] >> (k & 31)) & 1u;
    }
    __host__ __device__ void add(int n) {
        int k = n - lo;
        w[k >> 5] |= 1u << (k & 31);
    }
};

// The same set for windows of at most 32 sizes: one register instead of a bitmap in local memory.
struct SeenSmall {
    unsigned int w;
    int lo, hi;
    __host__ __device__ void reset(int lo_, int hi_) { lo = lo_, hi = hi_, w = 0u; }
    __host__ __device__ bool inside(int n) const { return n >= lo && n <= hi; }
    __host__ __device__ bool has(int n) const { return inside(n) && ((w >> (n - lo)) & 1u); }
    __host__ __device__ void add(int n) { w |= 1u << (n - lo); }
};

// The stack walk of the search (repeats.py:100-151) over a table of the sizes [n_lo, n_hi].  window(lo, hi) scores the
// sizes lo..hi in order: it adds those not yet in `seen` to it, counts them in n_scored (the count max_iters limits)
// and returns the size the climb moves to.  Returns the status: 0 ok, 1 a window left the table, 2 nothing scored.
// narrow = the search-policy switches (tie_flags bits 2-3, STRK_SEARCH_* in the header): the Rust body of this search
// is not in the reference tree and repeat_count_params.py:13 says the range "can be narrowed within the
// get_repeat_count fn".  0 = the in-tree statement (range fixed); the two narrowing hypotheses only ever shrink the
// windows, so the score table of a pass always covers them.
template <typename Seen, typename Window>
__host__ __device__ __forceinline__ int climb(int n_lo, int n_hi, int start_count, int max_iters, int range, int step,
                                              int narrow, Seen &seen, const int &n_scored, Window window) {
    seen.reset(n_lo, n_hi);
    int st_size[4], st_dir[4];
    int top = 0;
    st_size[top] = start_count - step, st_dir[top++] = -1;
    st_size[top] = start_count + step, st_dir[top++] = 1;
    st_size[top] = start_count, st_dir[top++] = 0;
    while (top > 0 && n_scored < max_iters) {
        --top;
        const int size = st_size[top], dir = st_dir[top];
        if (size < 0) continue;
        const bool wide = step > range;
        int lo = size - ((dir < 1 || wide) ? range : 0);
        if (lo < 0) lo = 0;
        const int hi = size + ((dir > -1 || wide) ? range : 0);
        // the window and the table are both contiguous: a window with a size outside the table has an end outside it
        if (!seen.inside(lo) || !seen.inside(hi)) return 1;
        if ((narrow & 4) && range > 1) range = 1;          // STRK_SEARCH_NARROW_FIRST: after the first window
        if ((narrow & 8) && range > 1) range = range / 2;  // STRK_SEARCH_NARROW_HALVE: after every window
        const int mv_size = window(lo, hi);
        // at most one of the two pushes can fire, so the stack never exceeds 3 entries
        if (mv_size > size) {
            const int new_rc = mv_size + step;
            if (!seen.has(new_rc) && new_rc >= 0) st_size[top] = new_rc, st_dir[top++] = 1;
        }
        if (mv_size < size) {
            const int new_rc = mv_size - step;
            if (!seen.has(new_rc) && new_rc >= 0) st_size[top] = new_rc, st_dir[top++] = -1;
        }
    }
    return n_scored ? 0 : 2;
}

// Single-score search (read path).  table[n - n_lo] for n in [n_lo, n_hi].
template <typename Seen>
__host__ __device__ inline ClimbResult climb_single(const int *table, int n_lo, int n_hi, int start_count,
                                                    int max_iters, int range, int step, int tie_flags,
                                                    Seen &seen) {
    ClimbResult res = {0, 0, 0, 0, 0.0, 0x7fffffff, -1};
    res.status = climb(n_lo, n_hi, start_count, max_iters, range, step, tie_flags & 12, seen, res.n_explored,
                       [&](int lo, int hi) {
        res.lo_touched = lo < res.lo_touched ? lo : res.lo_touched;
        res.hi_touched = hi > res.hi_touched ? hi : res.hi_touched;
        bool have = false;
        int mv_size = 0, mv_score = 0;
        for (int i = lo; i <= hi; ++i) {
            const int sc = table[i - n_lo];
            if (!seen.has(i)) {
                seen.add(i);
                // final pick = first-inserted maximum (repeats.py:154) unless STRK_TIE_FINAL_LAST
                if (!res.n_explored || sc > res.best_score || ((tie_flags & 2) && sc == res.best_score)) {
                    res.best_n = i;
                    res.best_score = sc;
                }
                ++res.n_explored;
                res.sum_n += (double)i;
            }
            // the move = first maximum of the window unless STRK_TIE_WINDOW_LAST
            if (!have || sc > mv_score || ((tie_flags & 1) && sc == mv_score)) {
                have = true;
                mv_size = i;
                mv_score = sc;
            }
        }
        return mv_size;
    });
    return res;
}

struct RefClimbResult {
    int l_offset, r_offset, n_offset_scores;
    int status;
};

// Dual-score search of get_ref_repeat_count (repeats.py:100-169).  tab[k] for k = n - n_lo holds the
// packed ARGMAX keys: fwd at tab[k], rev at tab[W + k]; score = key >> 32,
// end_query = 0x7fffffff - (key & 0xffffffff) - 1.
__host__ __device__ inline void ref_unpack(long long key, int &score, int &end_query) {
    score = (int)(key >> 32);
    end_query = 0x7fffffff - (int)(unsigned)(key & 0xffffffffll) - 1;
}

__host__ __device__ inline RefClimbResult climb_ref(const long long *tab, int n_lo, int n_hi, int start_count,
                                                   int max_iters, int range, int step, int n_fl, int n_fr,
                                                   int ref_size, int vcf_anchor_size, SeenSet &seen) {
    RefClimbResult res = {0, 0, 0, 0};
    const int W = n_hi - n_lo + 1;
    int bf_score = 0, bf_adj = 0, br_score = 0, br_adj = 0;
    res.status = climb(n_lo, n_hi, start_count, max_iters, range, step, 0, seen, res.n_offset_scores,
                       [&](int lo, int hi) {
        bool have = false;
        int mv_size = 0, mv_s = 0, mv_a = 0;
        // max((*fwd_scores, *rev_scores), key=(score, adj)): first maximal, fwd entries first (:135)
        for (int pass = 0; pass < 2; ++pass) {
            for (int i = lo; i <= hi; ++i) {
                int fs, fe, rs, re;
                ref_unpack(tab[i - n_lo], fs, fe);
                ref_unpack(tab[W + i - n_lo], rs, re);
                const int r_adj = fe + 1 - n_fl - ref_size;  // :34
                const int l_adj = re + 1 - n_fr - ref_size;  // :41
                if (!seen.has(i)) {
                    seen.add(i);
                    const bool first = res.n_offset_scores++ == 0;
                    if (first || fs > bf_score) bf_score = fs, bf_adj = r_adj;  // :154
                    if (first || rs > br_score) br_score = rs, br_adj = l_adj;  // :156
                }
                const int s = pass == 0 ? fs : rs, a = pass == 0 ? r_adj : l_adj;
                if (!have || s > mv_s || (s == mv_s && a > mv_a)) {
                    have = true;
                    mv_size = i;
                    mv_s = s;
                    mv_a = a;
                }
            }
        }
        return mv_size;
    });
    if (res.status) return res;
    res.l_offset = br_adj;  // :161
    res.r_offset = bf_adj;  // :162
    if (res.l_offset >= n_fl - vcf_anchor_size) res.l_offset = 0;  // :164-167
    if (res.r_offset >= n_fr) res.r_offset = 0;                    // :168-169
    return res;
}

// What the read loop needs of read r: its table row, estimate and lengths.
struct ReadRow {
    const int *row;
    int est, n_fl, n_tr, n_fr;
};

// Row source of replay_reads_kernel: the row of the read's slot (table + slot * W), or, when rep != nullptr (first
// pass only, slot == read), the row of read rep[r], whose table identical reads share.
struct GlobalRows {
    const int *table;
    int W;
    const int *rep, *est_cn, *lens;
    __device__ __forceinline__ ReadRow load(long long r, long long slot) const {
        return {table + (size_t)(rep ? (long long)rep[r] : slot) * (size_t)W, est_cn[r], lens[3 * r], lens[3 * r + 1],
                lens[3 * r + 2]};
    }
    __device__ __forceinline__ void begin(long long, long long, long long) {}
    __device__ __forceinline__ ReadRow next(long long r, long long, long long slot) { return load(r, slot); }
};

// Row source of replay_reads_small_kernel (W <= REPLAY_WMAX: every first pass).  The search reads a dozen table entries
// per read one after the other, each a trip to L2 (~4 us per read, 0.11 ms for a 30-read locus whatever the batch
// size): here read r is searched on a copy of its row in the thread's stripe of shared memory (stride REPLAY_WMAX + 1
// words: conflict-free) while the row, estimate and lengths of read r + 1 are fetched as independent loads.
#define REPLAY_WMAX 20
#define REPLAY_THREADS 128
struct StagedRows {
    GlobalRows src;
    int *stripe;
    int nrow[REPLAY_WMAX];
    ReadRow nxt;
    __device__ __forceinline__ void fetch(long long r, long long slot) {
        nxt = src.load(r, slot);
#pragma unroll
        for (int k = 0; k < REPLAY_WMAX; ++k) nrow[k] = k < src.W ? nxt.row[k] : 0;
    }
    __device__ __forceinline__ void begin(long long r0, long long r1, long long slot) {
        if (r0 < r1) fetch(r0, slot);
    }
    __device__ __forceinline__ ReadRow next(long long r, long long r1, long long slot) {
#pragma unroll
        for (int k = 0; k < REPLAY_WMAX; ++k) stripe[k] = nrow[k];
        ReadRow cur = nxt;
        cur.row = stripe;
        if (r + 1 < r1) fetch(r + 1, slot + 1);  // before the search of read r, which it overlaps
        return cur;
    }
};

// Locus q of a replay pass, one thread per locus: the read loop of call_locus.py:1129-1161 over the score tables.
//   window of a read = strk_slot_window, the table planner's; hint != nullptr: per locus {smallest, largest} offset
//   fraction seen at a miss, and a locus that misses adds the fraction it missed at
//   miss_count[0] += loci whose search left the window; miss_count[2] += loci that stayed inside it but went
//   beyond est +- wd, i.e. that only the wide_short margin saved from a second pass
//   locus_ids == nullptr: locus q is q and its slots are read_begin[q]..; otherwise the widening
//   pass lists the loci to redo and slot_begin[q] is the first slot of locus_ids[q].
template <typename Seen, typename Rows>
__device__ __forceinline__ void replay_locus(int q, Rows &rows, int wd, int wide_short, const int *locus_ids,
                                             const long long *slot_begin, const long long *read_begin,
                                             const int *motif_len, int max_iters, int range, int step, int tie_flags,
                                             int *out, unsigned char *locus_status, unsigned int *miss_count,
                                             double *ref_cells, double *hint) {
    const int locus = locus_ids ? locus_ids[q] : q;
    const long long r0 = read_begin[locus], r1 = read_begin[locus + 1];
    long long slot = locus_ids ? slot_begin[q] : r0;
    // a locus' hint changes only at its miss, which ends its loop
    double *h = hint ? hint + 2 * (size_t)locus : nullptr;
    double hl[2] = {0.0, 0.0};
    if (h) hl[0] = h[0], hl[1] = h[1];
    Seen seen;
    double frac = 0.0;  // read_offset_frac_from_starting_guess (:1079)
    double cells = 0.0;
    const int m = motif_len[locus];
    int status = 0;
    bool margin_used = false;
    rows.begin(r0, r1, slot);
    for (long long r = r0; r < r1; ++r, ++slot) {
        const ReadRow rd = rows.next(r, r1, slot);
        const int est = rd.est;
        int read_sc = est;
        const int off = (int)rint(frac * (double)read_sc);  // round(), :1130
        if (off < -read_sc)
            frac = 0.0;  // :1133
        else
            read_sc += off;  // :1136
        int n_lo, n_hi;
        strk_slot_window(est, m, wd, wide_short, h ? hl : nullptr, n_lo, n_hi);
        const ClimbResult cr = climb_single(rd.row, n_lo, n_hi, read_sc, max_iters, range, step, tie_flags, seen);
        if (cr.status) {
            status = cr.status;
            if (h && cr.status == 1) {  // where the next pass has to look: the fraction this read started from
                const double fr_used = read_sc == est ? 0.0 : frac;
                h[0] = fr_used < hl[0] ? fr_used : hl[0];
                h[1] = fr_used > hl[1] ? fr_used : hl[1];
            }
            break;
        }
        margin_used |= cr.lo_touched < est - wd || cr.hi_touched > est + wd;
        *(int4 *)(out + 4 * r) = make_int4(cr.best_n, cr.best_score, cr.n_explored, read_sc);
        frac += (double)(cr.best_n - read_sc) / (double)(cr.best_n > 1 ? cr.best_n : 1);  // :1161
        const double n1 = (double)(rd.n_fl + rd.n_tr + rd.n_fr);
        cells += n1 * ((double)cr.n_explored * (double)(rd.n_fl + rd.n_fr) + (double)m * cr.sum_n);
    }
    locus_status[locus] = (unsigned char)status;
    if (status) {
        atomicAdd(miss_count, 1u);
    } else {
        atomicAdd(ref_cells, cells);
        if (margin_used) atomicAdd(miss_count + 2, 1u);
    }
}

__global__ void replay_reads_kernel(const int *__restrict__ table, int W, int wd, int wide_short,
                                    const int *__restrict__ locus_ids,
                                    const long long *__restrict__ slot_begin, int n_list,
                                    const long long *__restrict__ read_begin, const int *__restrict__ est_cn,
                                    const int *__restrict__ lens, const int *__restrict__ motif_len, int max_iters,
                                    int range, int step, int tie_flags, int *__restrict__ out,
                                    unsigned char *__restrict__ locus_status, unsigned int *miss_count,
                                    double *ref_cells, const int *__restrict__ rep, double *__restrict__ hint = nullptr) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n_list) return;
    GlobalRows rows = {table, W, rep, est_cn, lens};
    replay_locus<SeenSet>(q, rows, wd, wide_short, locus_ids, slot_begin, read_begin, motif_len, max_iters, range, step,
                          tie_flags, out, locus_status, miss_count, ref_cells, hint);
}

__global__ void __launch_bounds__(REPLAY_THREADS)
    replay_reads_small_kernel(const int *__restrict__ table, int W, int wd, int wide_short,
                              const int *__restrict__ locus_ids, const long long *__restrict__ slot_begin, int n_list,
                              const long long *__restrict__ read_begin, const int *__restrict__ est_cn,
                              const int *__restrict__ lens, const int *__restrict__ motif_len, int max_iters, int range,
                              int step, int tie_flags, int *__restrict__ out, unsigned char *__restrict__ locus_status,
                              unsigned int *miss_count, double *ref_cells, const int *__restrict__ rep,
                              double *__restrict__ hint = nullptr) {
    __shared__ int stripes[REPLAY_THREADS * (REPLAY_WMAX + 1)];
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n_list) return;
    StagedRows rows;
    rows.src = {table, W, rep, est_cn, lens};
    rows.stripe = stripes + threadIdx.x * (REPLAY_WMAX + 1);
    replay_locus<SeenSmall>(q, rows, wd, wide_short, locus_ids, slot_begin, read_begin, motif_len, max_iters, range,
                            step, tie_flags, out, locus_status, miss_count, ref_cells, hint);
}

// Builds the family descriptors of a pass on the device (no descriptor H2D traffic).
//   read_ids == nullptr: slot s is read s.
__global__ void plan_reads_kernel(const int *__restrict__ read_ids, long long n_slots,
                                  const unsigned long long *__restrict__ seq_off, const int *__restrict__ lens,
                                  const int *__restrict__ est_cn, const int *__restrict__ read_locus,
                                  const unsigned long long *__restrict__ motif_off, const int *__restrict__ motif_len,
                                  int wd, int wide_short, int W, FamDesc *__restrict__ fams, double *exec_cells,
                                  const int *__restrict__ rep, const double *__restrict__ hint = nullptr,
                                  unsigned int *w_needed = nullptr) {
    // w_needed != nullptr: only measure -- the widest window of the pass (atomicMax), no descriptor is written
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    double cells = 0.0;
    if (s < n_slots) {
    const long long r = read_ids ? read_ids[s] : s;
    const int locus = read_locus[r];
    FamDesc f;
    f.db_off = seq_off[r];
    f.motif_off = motif_off[locus];
    f.out_off = (unsigned long long)s * (unsigned long long)W;
    f.n_fl = lens[3 * r];
    f.n_tr = lens[3 * r + 1];
    f.n_fr = lens[3 * r + 2];
    f.m = motif_len[locus];
    const int est = est_cn[r];
    strk_slot_window(est, f.m, wd, wide_short, hint ? hint + 2 * (size_t)locus : nullptr, f.n_lo, f.n_hi);
    if (w_needed) {
        atomicMax(w_needed, (unsigned int)(f.n_hi - f.n_lo + 1));
    } else {
        fams[s] = f;
        // executed DP cells: one forward sweep over fl + motif*n_hi plus one backward sweep over fr
        if (!rep || rep[r] == (int)r)  // a read that shares another read's table executes no cells
            cells = (double)(f.n_fl + f.n_tr + f.n_fr) * ((double)f.n_fl + (double)f.m * (double)f.n_hi + (double)f.n_fr);
    }
    }
    for (int o = 16; o > 0; o >>= 1) cells += __shfl_down_sync(0xffffffffu, cells, o);
    if ((threadIdx.x & 31) == 0 && cells > 0.0) atomicAdd(exec_cells, cells);
}
