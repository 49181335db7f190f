// ref_path.cuh -- device-side planning and replay of get_ref_repeat_count (strkit/call/repeats.py:73-192),
// one thread per locus.  Phase 1: the boundary search over the two sg_qe tables (score_ref_boundaries, :23-43;
// climb_ref in replay.cuh restates :100-169) -> l_offset / r_offset.  Phase 2 re-uses the read-path batch machinery
// on the adjusted flanks (:171-188).  The host only sees counters, the results and the flags of the loci whose search
// left its window (those it finishes itself).
#pragma once
#include "replay.cuh"
#include "strk_common.cuh"

// Family descriptors of the boundary tables of a pass.  ids == nullptr: locus q is q.
// Window of locus l = [max(lo_min, start - wd[l]), start + wd[l]]; its table region = 2 * stride_w keys at 2 * q * stride_w.
__global__ void ref_plan1_kernel(const int *__restrict__ ids, int n, const unsigned long long *__restrict__ seq_off,
                                 const int *__restrict__ lens, const int *__restrict__ start, const int *__restrict__ wd,
                                 const unsigned long long *__restrict__ motif_off, const int *__restrict__ motif_len,
                                 int stride_w, FamDesc *__restrict__ fams, const unsigned int *__restrict__ n_dev = nullptr) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (n_dev && (unsigned)n > *n_dev) n = (int)*n_dev;  // list length produced on the device; n is its upper bound
    if (q >= n) return;
    const int l = ids ? ids[q] : q;
    FamDesc f;
    f.db_off = seq_off[l];
    f.motif_off = motif_off[l];
    f.n_fl = lens[3 * l], f.n_tr = lens[3 * l + 1], f.n_fr = lens[3 * l + 2], f.m = motif_len[l];
    // size 0 with an empty flank would be an empty candidate; the replay reports it if it gets there
    const int lo_min = (f.n_fl == 0 || f.n_fr == 0) ? 1 : 0;
    const int lo = start[l] - wd[l];
    f.n_lo = lo > lo_min ? lo : lo_min;
    const int hi = start[l] + wd[l];
    f.n_hi = hi > f.n_lo ? hi : f.n_lo;
    f.out_off = (unsigned long long)q * (unsigned long long)stride_w;
    fams[q] = f;
}

// counters: [0] loci to redo with a wider window (appended to again_ids), [1] 1 + smallest locus that scored no
// size (0 = none), [2] 1 + smallest locus that left the widest window (0 = none)
__global__ void ref_replay1_kernel(const int *__restrict__ ids, int n, const long long *__restrict__ tab,
                                   const FamDesc *__restrict__ fams, const int *__restrict__ start,
                                   const int *__restrict__ rc, const int *__restrict__ ref_size, int vcf_anchor_size,
                                   int wd_max, int *__restrict__ wd, int *__restrict__ l_off, int *__restrict__ r_off,
                                   int *__restrict__ n_off, int *__restrict__ again_ids, unsigned int *counters,
                                   const unsigned int *__restrict__ n_dev = nullptr) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (n_dev && (unsigned)n > *n_dev) n = (int)*n_dev;
    if (q >= n) return;
    const int l = ids ? ids[q] : q;
    const FamDesc f = fams[q];
    SeenSet seen;
    const RefClimbResult cr = climb_ref(tab + 2 * f.out_off, f.n_lo, f.n_hi, start[l], rc[3 * l], rc[3 * l + 1],
                                        rc[3 * l + 2], f.n_fl, f.n_fr, ref_size[l], vcf_anchor_size, seen);
    if (cr.status == 1) {
        n_off[l] = -1;  // not final yet (ref_assemble_kernel flags the locus for the host; a wider pass overwrites it)
        if (wd[l] >= wd_max) {
            atomicMax(&counters[2], 0x7fffffffu - (unsigned)l);
            return;
        }
        const int w4 = wd[l] * 4;
        wd[l] = w4 < wd_max ? w4 : wd_max;
        again_ids[atomicAdd(&counters[0], 1u)] = l;
        return;
    }
    if (cr.status == 2) {
        atomicMax(&counters[1], 0x7fffffffu - (unsigned)l);
        return;
    }
    l_off[l] = cr.l_offset;
    r_off[l] = cr.r_offset;
    n_off[l] = cr.n_offset_scores;
}

// Phase 2 inputs of the loci of one search-parameter tier: the tract extended by what phase 1 moved out of the
// flanks (repeats.py:171-176), start = round((start * m + moved) / m) (:180-186), one "read" per locus.
__global__ void ref_plan2_kernel(const int *__restrict__ ids, int n, const unsigned long long *__restrict__ seq_off,
                                 const int *__restrict__ lens, const int *__restrict__ start,
                                 const unsigned long long *__restrict__ motif_off, const int *__restrict__ motif_len,
                                 const int *__restrict__ l_off, const int *__restrict__ r_off,
                                 unsigned long long *__restrict__ seq_off2, int *__restrict__ lens2, int *__restrict__ est2,
                                 unsigned long long *__restrict__ motif_off2, int *__restrict__ motif_len2,
                                 long long *__restrict__ read_begin2, int *__restrict__ read_locus2 = nullptr) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q == 0) read_begin2[n] = n;
    if (q >= n) return;
    const int l = ids ? ids[q] : q;  // ids == nullptr: every locus, in order
    if (read_locus2) read_locus2[q] = q;
    const int mov_l = l_off[l] > 0 ? l_off[l] : 0, mov_r = r_off[l] > 0 ? r_off[l] : 0;
    const int n1 = lens[3 * l] + lens[3 * l + 1] + lens[3 * l + 2];
    const int nfl = lens[3 * l] - mov_l, nfr = lens[3 * l + 2] - mov_r;
    const int m = motif_len[l];
    seq_off2[q] = seq_off[l];
    lens2[3 * q] = nfl;
    lens2[3 * q + 1] = n1 - nfl - nfr;
    lens2[3 * q + 2] = nfr;
    // round() of the float quotient: banker's rounding (repeats.py:182)
    est2[q] = (int)rint(((double)start[l] * (double)m + (double)(mov_l + mov_r)) / (double)m);
    motif_off2[q] = motif_off[l];
    motif_len2[q] = m;
    read_begin2[q] = q;
}

// The 8 result ints of the loci of a phase 2 pass (slot q = locus ids[q]; ids == nullptr: locus q), assembled on the
// device, and their redo flags: the host finishes the loci whose phase 1 is not final or whose phase 2 search failed.
//   out[8l..] = {cn, score, l_offset, r_offset, n_offset_scores (-1: phase 1 not final), n_iters_final, new fl, new fr}
__global__ void ref_assemble_kernel(const int *__restrict__ ids, int n, const int *__restrict__ res4,
                                    const unsigned char *__restrict__ status, const int *__restrict__ lens,
                                    const int *__restrict__ l_off, const int *__restrict__ r_off,
                                    const int *__restrict__ n_off, int *__restrict__ out, unsigned char *__restrict__ redo) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const int l = ids ? ids[q] : q;
    const int lo = l_off[l], ro = r_off[l];
    int *o = out + 8 * (size_t)l;
    const bool ok = status[q] == 0;
    o[0] = ok ? res4[4 * q] : 0;
    o[1] = ok ? res4[4 * q + 1] : 0;
    o[2] = lo;
    o[3] = ro;
    o[4] = n_off[l];
    o[5] = ok ? res4[4 * q + 2] : 0;
    o[6] = lens[3 * l] - (lo > 0 ? lo : 0);
    o[7] = lens[3 * l + 2] - (ro > 0 ? ro : 0);
    redo[l] = !ok || n_off[l] < 0;
}

__global__ void ref_clamp_count_kernel(unsigned int *count, unsigned int cap) {
    if (threadIdx.x == 0 && blockIdx.x == 0 && *count > cap) *count = cap;
}
