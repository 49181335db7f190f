// plan.cuh -- device-side validation and work planning of a batch.
//
// The host batcher hands over raw arrays; everything per-read (argument checks, locus index of each read,
// kernel / rows-per-lane class, the segmented work order, scratch sizing maxima) is computed here so that
// the host-buffer C-ABI call costs one H2D copy plus a few microsecond-scale kernels, not several passes
// over millions of reads on one CPU core.
#pragma once
#include "dp_packed.cuh"
#include "strk_common.cuh"

// ---- the rules of a batch: the device planner below, the host planner and the direct entry points (api.cu) call these

enum PlanError {
    PLAN_ERR_NEG_LEN = 1, PLAN_ERR_EMPTY = 2, PLAN_ERR_TOO_LONG = 3, PLAN_ERR_PAST_ARENA = 4, PLAN_ERR_EST = 5,
    PLAN_ERR_MOTIF_EMPTY = 6, PLAN_ERR_MOTIF_PAST_ARENA = 7, PLAN_ERR_READ_BEGIN = 8
};

// A locus whose reads are [r0, r1) of n_reads and whose motif is motif_len bases at motif_off: 0, or its PlanError.
__host__ __device__ inline int strk_check_locus(long long r0, long long r1, long long n_reads, unsigned long long motif_off,
                                                int motif_len, unsigned long long arena_bytes) {
    if (r1 < r0 || r0 < 0 || r1 > n_reads) return PLAN_ERR_READ_BEGIN;
    if (motif_len <= 0) return PLAN_ERR_MOTIF_EMPTY;
    if (motif_off > arena_bytes || (unsigned long long)motif_len > arena_bytes - motif_off) return PLAN_ERR_MOTIF_PAST_ARENA;
    return 0;
}

// A read of flanks fl / fr around a tract of tr bases at seq_off: 0, or its PlanError.
__host__ __device__ inline int strk_check_read(int fl, int tr, int fr, unsigned long long seq_off,
                                               unsigned long long arena_bytes) {
    if (fl < 0 || tr < 0 || fr < 0) return PLAN_ERR_NEG_LEN;
    const long long n1 = (long long)fl + tr + fr;
    if (n1 <= 0) return PLAN_ERR_EMPTY;
    if (n1 > (1 << 24)) return PLAN_ERR_TOO_LONG;
    if (seq_off > arena_bytes || (unsigned long long)n1 > arena_bytes - seq_off) return PLAN_ERR_PAST_ARENA;  // (no wrap-around)
    return 0;
}

// A start estimate of est copies of an m-base motif: candidate columns are counted in 64 bits, so that a garbage
// estimate cannot size scratch.
__host__ __device__ inline int strk_check_est(int est, int m) {
    return est < 0 || est > (1 << 22) || (long long)m * (long long)est > (1ll << 24) ? PLAN_ERR_EST : 0;
}

// Scratch of the general kernel (dp_general.cuh) for a set of reads: the backward column of the longest db and, when
// a read takes more than one strip, the boundary row between strips: the longest candidate prefix, plus wd copies of
// the largest motif for the sizes a window adds.  No constructor, so that it can live in shared memory and in the
// zero-filled PlanStats: start from GenExtent{}.
struct GenExtent {
    int max_n1;   // longest db
    int mb_cols;  // reads of more than one strip: max of max(fl, fr) + m * copies
    int mb_m;     //                               max motif length
    __host__ __device__ void add(int fl, int fr, int n1, int m, int copies) {
        if (n1 > max_n1) max_n1 = n1;
        if (n1 > GEN_STRIP_ROWS) {
            const int cols = (fl > fr ? fl : fr) + m * copies;
            if (cols > mb_cols) mb_cols = cols;
            if (m > mb_m) mb_m = m;
        }
    }
    __host__ __device__ int b_len() const { return max_n1 + 2; }
    __host__ __device__ int rowlen(int wd) const { return max_n1 > GEN_STRIP_ROWS ? mb_cols + mb_m * wd + 2 : 2; }
};

struct PlanStats {
    unsigned long long first_error;  // (index << 8 | kind), smallest wins; ~0 = none
    unsigned bin_cnt[STRK_PK_NBIN];  // reads per class: [0] general kernel only, [R] packed kernel with R rows per lane
    unsigned bin_cursor[STRK_PK_NBIN];
    int bin_mmax[STRK_PK_NBIN], bin_flank[STRK_PK_NBIN];
    GenExtent ext;   // of the valid reads
    unsigned n_dup;  // reads that share an earlier read's table (dedupe.cuh)
};

// Rows-per-lane class of the packed kernel for a window of flanks fl / fr around a tract of tr bases and a motif of m
// bases; 0 = the general kernel only (too long, a flank it cannot stage, or a motif profile wider than 128 rows).
// Callers add their own gates: the matrix (packed_ok) and the window of candidate sizes.
__host__ __device__ inline int strk_pk_class(int fl, int tr, int fr, int m) {
    const int R = strk_pick_rows_packed(fl + tr + fr + 1);
    if (fl < 1 || fr < 1 || fl > PK_FLANK_MAX || fr > PK_FLANK_MAX || m * R > 128 || m <= 0) return 0;
    return R;
}

__device__ __forceinline__ void plan_report(PlanStats *st, long long index, int kind) {
    atomicMin(&st->first_error, ((unsigned long long)index << 8) | (unsigned long long)kind);
}

// one thread per locus: motif checks, read_begin monotonicity, read -> locus map
__global__ void plan_loci_kernel(const long long *__restrict__ read_begin, long long n_loci, long long n_reads,
                                 const unsigned long long *__restrict__ motif_off, const int *__restrict__ motif_len,
                                 unsigned long long arena_bytes, int *__restrict__ read_locus, PlanStats *st) {
    const long long l = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= n_loci) return;
    const long long r0 = read_begin[l], r1 = read_begin[l + 1];
    const int kind = strk_check_locus(r0, r1, n_reads, motif_off[l], motif_len[l], arena_bytes);
    if (kind) {
        plan_report(st, l, kind);
        return;
    }
    for (long long r = r0; r < r1; ++r) read_locus[r] = (int)l;
}

// one thread per read: argument checks, class, per-class histogram and maxima
__global__ void plan_reads_scan_kernel(const unsigned long long *__restrict__ seq_off, const int *__restrict__ lens,
                                       const int *__restrict__ est_cn, const int *__restrict__ read_locus,
                                       const int *__restrict__ motif_len, long long n_reads,
                                       unsigned long long arena_bytes, int packed_ok, unsigned char *__restrict__ bin,
                                       PlanStats *st) {
    __shared__ unsigned s_cnt[STRK_PK_NBIN];
    __shared__ int s_mmax[STRK_PK_NBIN], s_flank[STRK_PK_NBIN];
    __shared__ GenExtent s_ext;
    if (threadIdx.x < STRK_PK_NBIN) s_cnt[threadIdx.x] = 0, s_mmax[threadIdx.x] = 0, s_flank[threadIdx.x] = 0;
    if (threadIdx.x == 0) s_ext = GenExtent{};
    __syncthreads();
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n_reads) {
        const int fl = lens[3 * r], tr = lens[3 * r + 1], fr = lens[3 * r + 2];
        const int m = motif_len[read_locus[r]], est = est_cn[r];
        int kind = strk_check_read(fl, tr, fr, seq_off[r], arena_bytes);
        if (!kind) kind = strk_check_est(est, m);
        int b = 0;
        if (kind)
            plan_report(st, r, kind);
        else {
            b = packed_ok ? strk_pk_class(fl, tr, fr, m) : 0;
            if (b) {
                atomicMax(&s_mmax[b], m);
                atomicMax(&s_flank[b], fl > fr ? fl : fr);
            }
            GenExtent e = {};
            e.add(fl, fr, fl + tr + fr, m, est);
            atomicMax(&s_ext.max_n1, e.max_n1);
            if (e.mb_m) {
                atomicMax(&s_ext.mb_cols, e.mb_cols);
                atomicMax(&s_ext.mb_m, e.mb_m);
            }
        }
        bin[r] = (unsigned char)b;
        atomicAdd(&s_cnt[b], 1u);
    }
    __syncthreads();
    if (threadIdx.x < STRK_PK_NBIN) {
        if (s_cnt[threadIdx.x]) atomicAdd(&st->bin_cnt[threadIdx.x], s_cnt[threadIdx.x]);
        if (s_mmax[threadIdx.x]) atomicMax(&st->bin_mmax[threadIdx.x], s_mmax[threadIdx.x]);
        if (s_flank[threadIdx.x]) atomicMax(&st->bin_flank[threadIdx.x], s_flank[threadIdx.x]);
    }
    if (threadIdx.x == 0) {
        atomicMax(&st->ext.max_n1, s_ext.max_n1);
        if (s_ext.mb_cols) atomicMax(&st->ext.mb_cols, s_ext.mb_cols);
        if (s_ext.mb_m) atomicMax(&st->ext.mb_m, s_ext.mb_m);
    }
}

// segmented work order: class k occupies order[bin_off[k] .. bin_off[k] + bin_cnt[k])
//   rep != nullptr: reads with rep[r] != r share an earlier read's table and get no work item
__global__ void plan_reads_scatter_kernel(const unsigned char *__restrict__ bin, long long n_reads,
                                          const unsigned *__restrict__ bin_off, PlanStats *st, int *__restrict__ order,
                                          const int *__restrict__ rep) {
    __shared__ unsigned s_cnt[STRK_PK_NBIN], s_base[STRK_PK_NBIN];
    if (threadIdx.x < STRK_PK_NBIN) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int b = 0;
    unsigned local = 0;
    const bool mine = r < n_reads && (!rep || rep[r] == (int)r);
    if (mine) {
        b = bin[r];
        local = atomicAdd(&s_cnt[b], 1u);
    }
    __syncthreads();
    if (threadIdx.x < STRK_PK_NBIN && s_cnt[threadIdx.x]) s_base[threadIdx.x] = atomicAdd(&st->bin_cursor[threadIdx.x], s_cnt[threadIdx.x]);
    __syncthreads();
    if (mine) order[bin_off[b] + s_base[b] + local] = (int)r;
}

// Nibble-packed host arenas (STRK_ARENA_NIBBLE): two symbols per byte, low nibble first, code = index into
// "ACGTRYSWKMBDHVNX" (align_matrix.py:25-26).  Halves the H2D bytes of a block; this kernel expands the packed copy
// into the byte-per-symbol arena every DP kernel stages from, right after the copy lands.  One 128-bit load and two
// 128-bit stores per thread, coalesced; memory-bound (0.45 GB per million reads, < 0.1 ms at HBM speed).
__global__ void expand_nibbles_kernel(const uint4 *__restrict__ packed, unsigned long long n_bytes,
                                      unsigned char *__restrict__ out) {
    __shared__ unsigned char lut[16];
    if (threadIdx.x < 16) lut[threadIdx.x] = (unsigned char)"ACGTRYSWKMBDHVNX"[threadIdx.x];
    __syncthreads();
    const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned long long n_quads = n_bytes >> 4;
    if (i < n_quads) {
        const uint4 v = packed[i];
        const unsigned w[4] = {v.x, v.y, v.z, v.w};
        unsigned o[8];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const unsigned x = w[k] >> (16 * h);
                o[2 * k + h] = (unsigned)lut[x & 15u] | ((unsigned)lut[(x >> 4) & 15u] << 8) |
                               ((unsigned)lut[(x >> 8) & 15u] << 16) | ((unsigned)lut[(x >> 12) & 15u] << 24);
            }
        }
        uint4 *dst = (uint4 *)(out + 32ull * i);
        dst[0] = make_uint4(o[0], o[1], o[2], o[3]);
        dst[1] = make_uint4(o[4], o[5], o[6], o[7]);
    } else if (i == n_quads) {  // tail: fewer than 16 packed bytes
        const unsigned char *pb = (const unsigned char *)packed;
        for (unsigned long long b = n_quads << 4; b < n_bytes; ++b) {
            out[2 * b] = lut[pb[b] & 15u];
            out[2 * b + 1] = lut[pb[b] >> 4];
        }
    }
}
