// api.cu -- C ABI (include/strkit_b200.h), context and batch management, launch orchestration.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <vector>

#include "../../include/strkit_b200.h"
#include "dp_general.cuh"
#include "dp_packed.cuh"
#include "plan.cuh"
#include "dedupe.cuh"
#include "int_peak.cuh"
#include "replay.cuh"
#include "ref_path.cuh"
#include "strk_common.cuh"

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int set_err(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t e_ = (call);                                                                          \
        if (e_ != cudaSuccess)                                                                            \
            return set_err(STRK_ERR_CUDA, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__,            \
                           cudaGetErrorString(e_));                                                       \
    } while (0)

extern "C" const char *strk_last_error(void) { return g_err; }
extern "C" const char *strk_version(void) { return "strkit_b200 0.1 (sm_100a)"; }

extern "C" int strk_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

// ------------------------------------------------------------------------------------------------
// device buffer that only grows
// ------------------------------------------------------------------------------------------------
template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = n + n / 8 + 16;
        cudaError_t e = cudaMalloc((void **)&p, want * sizeof(T));
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

// One DP pass (launch_pass): the families, their table, and per rows-per-lane class k the device list of work items
// (0 = families only the general kernel takes) with the maxima the packed launch of class k sizes its tables by.
struct DpPass {
    const FamDesc *fams = nullptr;
    const unsigned char *arena = nullptr;
    void *table = nullptr;
    int ref_mode = 0;  // the families are reference windows and `table` holds the 64-bit boundary keys
    int b_len = 0, rowlen = 0;
    long long n_slots = 0;
    const int *list[STRK_PK_NBIN] = {nullptr};  // list[0] == nullptr: the families 0 .. cnt[0] - 1
    long long cnt[STRK_PK_NBIN] = {0};
    int flank[STRK_PK_NBIN] = {0}, mmax[STRK_PK_NBIN] = {0}, w[STRK_PK_NBIN] = {0};  // w: sizes of the widest window
};

// Work items of a DP pass binned by rows-per-lane class (0 = general kernel only), with the per-class maxima the packed
// launches size their tables by.
struct ClassLists {
    std::vector<int> items[STRK_PK_NBIN];
    std::vector<int> flat;  // every list, class after class: the host source of one H2D copy
    int mmax[STRK_PK_NBIN] = {0}, flank[STRK_PK_NBIN] = {0}, w_max[STRK_PK_NBIN] = {0};
    void clear() {
        for (int k = 0; k < STRK_PK_NBIN; ++k) items[k].clear(), mmax[k] = flank[k] = w_max[k] = 0;
    }
    void add(int k, int item) { items[k].push_back(item); }
    void add(int k, int item, int m, int fl, int fr, int w = 0) {
        items[k].push_back(item);
        mmax[k] = std::max(mmax[k], m);
        flank[k] = std::max(flank[k], std::max(fl, fr));
        w_max[k] = std::max(w_max[k], w);
    }
    // Queues the copy of the lists into `buf` on `st` and points the classes of `p` at the device segments, with these
    // maxima.  `flat` is read by the copy until `st` has passed it.
    int upload(DevBuf<int> &buf, cudaStream_t st, DpPass &p) {
        size_t at[STRK_PK_NBIN];
        flat.clear();
        for (int k = 0; k < STRK_PK_NBIN; ++k) {
            at[k] = flat.size();
            flat.insert(flat.end(), items[k].begin(), items[k].end());
        }
        if (buf.reserve(flat.size()) != cudaSuccess) {
            cudaGetLastError();
            return set_err(STRK_ERR_NOMEM, "cannot allocate the class lists of a pass");
        }
        CU(cudaMemcpyAsync(buf.p, flat.data(), flat.size() * sizeof(int), cudaMemcpyHostToDevice, st));
        for (int k = 0; k < STRK_PK_NBIN; ++k) {
            p.list[k] = buf.p + at[k], p.cnt[k] = (long long)items[k].size();
            p.flank[k] = flank[k], p.mmax[k] = mmax[k], p.w[k] = w_max[k];
        }
        return STRK_OK;
    }
};

// One search-parameter tier of a strk_ref_counts call (repeat_count_params.py:17-42): phase 2 runs once per tier
struct RefTier {
    int rc[3];             // max_iters, local search range, step size
    int wd2, W2;           // phase 2's first window: half-width, sizes
    std::vector<int> ids;  // its loci, ascending
    ClassLists classes;    // phase 2's classes over the tier's slots (unused when phase 1's lists serve)
};

// The reference path's per-locus state (strk_ref_counts), recycled across calls
struct RefBufs {
    DevBuf<unsigned char> arena;
    DevBuf<unsigned long long> seq_off, motif_off;
    DevBuf<int> lens, start, ref_size, rc, motif_len;  // the caller's arrays
    DevBuf<int> wd;                                    // half-width of each locus' next boundary window
    DevBuf<int> l_off, r_off, n_off;                   // phase 1 results
    DevBuf<int> ids_a, ids_b;                          // locus lists: pending loci of phase 1, the flagged loci of a tier
    DevBuf<int> tier_ids;                              // the loci of every tier, tier after tier
    DevBuf<int> lists;                                 // class lists of a packed pass
    DevBuf<unsigned int> cnt;                          // counters of ref_replay1_kernel: [0, 4) a pass, [4, 8) a second look
    DevBuf<int> out;                                   // the results, assembled on the device
    DevBuf<unsigned char> redo;                        // per locus: left to the host (a search left its window)
    // host sources of asynchronous copies: alive until the stream has passed them (one synchronisation per call)
    std::vector<int> h_wd;
    ClassLists classes;
    std::vector<RefTier> tiers;
    void release() {
        arena.release(), seq_off.release(), motif_off.release(), lens.release(), start.release(), ref_size.release();
        rc.release(), motif_len.release(), wd.release(), l_off.release(), r_off.release(), n_off.release();
        ids_a.release(), ids_b.release(), tier_ids.release(), lists.release(), cnt.release(), out.release(), redo.release();
    }
};

// The device counter words of a context (strk_ctx::d_queue, addressed through strk_ctx::counter)
enum CounterSlot : int {
    Q_GENERAL = 0,   // work queue of the general kernel
    Q_MISS = 1,      // loci whose search left the window (the replay kernels)
    Q_FALLBACK = 2,  // reads the packed kernel handed to the general kernel
    Q_MARGIN = 3,    // loci the wide_short margin saved (the replay kernels count them at Q_MISS + 2)
    Q_WIDEST = 6,    // the widest stretched window of a widening pass
    Q_INT_PEAK = 7,  // the output word of strk_measure_int_peak
    Q_CLASS = 8,     // + k: work queue of packed class k
};
static_assert(Q_FALLBACK == Q_MISS + 1 && Q_MARGIN == Q_MISS + 2, "strk_batch_run reads the three words in one copy");

struct strk_ctx {
    int device = 0;
    int n_sm = 0;
    // small passes: one side stream per rows-per-lane class, so the class launches (each under one wave) overlap
    cudaStream_t side[STRK_PK_NBIN] = {nullptr};
    cudaEvent_t side_ev[STRK_PK_NBIN] = {nullptr};
    cudaEvent_t fork_ev = nullptr;
    cudaStream_t stream = nullptr;
    // Uploads and planning kernels of strk_batch_fill run on a LOW-priority stream, the DP streams are created with the
    // greatest priority: in the streamed path the fill of block i + 1 (two contexts) shares the GPU with the DP kernels
    // of block i, and its large grids of short blocks (one warp per read) would otherwise take the slots every
    // finishing DP class frees before the next class' CTAs can.
    cudaStream_t fill_stream = nullptr;
    int prio_hi = 0;
    ScoreConsts h_consts;
    ScoreConsts *d_consts = nullptr;
    int gap = 5, end_flags = STRK_MODE_SG, tie_flags = 0;
    DevBuf<int> scratch;
    DevBuf<FamDesc> fams;
    DevBuf<int> table;
    DevBuf<long long> table64;
    DevBuf<int> list_a, list_b, list_d;  // widening-pass lists
    DevBuf<long long> list_c;
    DevBuf<int> fallback;            // reads the packed kernel handed to the general kernel
    DevBuf<uint4> pk_scratch;        // captured DP columns of the packed kernel (per resident warp)
    DevBuf<double> al_rep[3];        // allele calling: replicate means / weights / stdevs of one chunk of loci
    DevBuf<unsigned char> al_peaks;  //                 replicate peak counts
    // reference path (strk_ref_counts): per-locus state, and the one-read-per-locus batch of phase 2
    RefBufs ref;
    struct strk_batch *ref_batch = nullptr;
    DevBuf<int> al_i[12];            //                 per-read / per-locus integer arrays (recycled across calls)
    DevBuf<double> al_d[4];
    DevBuf<long long> al_rb;
    DevBuf<long long> al_doff;       //                 offsets of the deep loci's ragged values / CDF
    unsigned int *d_queue = nullptr;  // counter words (CounterSlot)
    unsigned int *counter(int slot) const { return d_queue + slot; }
    double *d_acc = nullptr;          // [0] ref cells, [1] executed cells
    PlanStats *d_plan = nullptr;      // device-side planning counters
    unsigned int *d_bin_off = nullptr;
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    double stats[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    struct strk_batch *reuse = nullptr;  // device buffers recycled by strk_count_reads
};

struct strk_batch {
    long long n_reads = 0, n_loci = 0;
    DevBuf<unsigned char> arena, status;
    DevBuf<uint4> arena4;  // nibble-packed copy as uploaded (STRK_ARENA_NIBBLE), expanded into `arena` on the device
    DevBuf<unsigned long long> seq_off, motif_off;
    DevBuf<int> lens, est, motif_len, read_locus, order, out;
    DevBuf<long long> read_begin;
    unsigned char *d_arena = nullptr;
    unsigned long long *d_seq_off = nullptr, *d_motif_off = nullptr;
    int *d_lens = nullptr, *d_est = nullptr, *d_motif_len = nullptr, *d_read_locus = nullptr, *d_order = nullptr;
    long long *d_read_begin = nullptr;
    int *d_out = nullptr;
    unsigned char *d_status = nullptr;
    // host mirror used by the widening passes (per locus, small); per-read planning happens on the device
    std::vector<long long> h_read_begin;
    DevBuf<unsigned char> bin;
    // identical reads of a locus share one table (dedupe.cuh): rep[r] = the read whose row r uses
    DevBuf<unsigned long long> hash;
    DevBuf<int> rep;
    DevBuf<double> hint;  // per locus {smallest, largest} carried-offset fraction seen at a window miss (strk_slot_window)
    int *d_rep = nullptr;
    long long n_dup = 0;
    GenExtent ext = {};  // the general kernel's scratch for these reads
    // first-window policy, carried from one block of loci to the next one filled into this object: 1 = short motifs
    // get the wider first window of strk_read_wd (set when a block sent > 2.5 % of its loci to a second pass,
    // cleared when < 1 % of a block's loci used the margin).  Speed only: results never depend on the window.
    int wide_short = 0;
    // work plan over h_order: [0, n_general) general-kernel-only reads, then one segment per packed R
    long long n_general = 0;
    long long bin_off[STRK_PK_NBIN] = {0}, bin_cnt[STRK_PK_NBIN] = {0};  // index R (0 = general kernel)
    int bin_mmax[STRK_PK_NBIN] = {0}, bin_flank[STRK_PK_NBIN] = {0};
    void release() {
        arena.release(), status.release(), seq_off.release(), motif_off.release(), lens.release(), est.release();
        motif_len.release(), read_locus.release(), order.release(), out.release(), read_begin.release();
        bin.release(), hash.release(), rep.release(), arena4.release(), hint.release();
    }
};

// ------------------------------------------------------------------------------------------------
// init / destroy
// ------------------------------------------------------------------------------------------------
static void build_lut(unsigned char lut[256]) {
    // parasail matrix_create mapper: alphabet "ACGTRYSWKMBDHVNX" (align_matrix.py:25), case-insensitive,
    // everything else -> the wildcard column (index 16)
    const char *alpha = "ACGTRYSWKMBDHVNX";
    for (int i = 0; i < 256; ++i) lut[i] = 16;
    for (int i = 0; i < 16; ++i) {
        lut[(unsigned char)alpha[i]] = (unsigned char)i;
        lut[(unsigned char)(alpha[i] - 'A' + 'a')] = (unsigned char)i;
    }
}

extern "C" int strk_destroy(strk_ctx *ctx);

extern "C" int strk_init(int device, const int8_t matrix[STRK_NSYM * STRK_NSYM], int gap_open, int gap_extend,
                         int end_flags, int tie_flags, strk_ctx **out) {
    if (!out || !matrix) return set_err(STRK_ERR_ARG, "strk_init: null argument");
    *out = nullptr;
    if (gap_open != gap_extend)
        return set_err(STRK_ERR_UNSUPPORTED,
                       "gap_open (%d) != gap_extend (%d): only the linear-gap case the reference uses "
                       "(indel_penalty for both, repeats.py:33) is implemented",
                       gap_open, gap_extend);
    if (gap_open < 1 || gap_open > 60) return set_err(STRK_ERR_ARG, "gap penalty %d out of range [1, 60]", gap_open);
    if (end_flags < 0 || end_flags > 15) return set_err(STRK_ERR_ARG, "end_flags %d out of range", end_flags);
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev == 0) {
        cudaGetLastError();
        return set_err(STRK_ERR_CUDA, "no CUDA device available (%s); strkit_b200 has no CPU fallback",
                       e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= n_dev) return set_err(STRK_ERR_ARG, "device %d out of range (%d devices)", device, n_dev);
    CU(cudaSetDevice(device));
    strk_ctx *ctx = new (std::nothrow) strk_ctx();
    if (!ctx) return set_err(STRK_ERR_NOMEM, "out of host memory");
    // any failure below releases what has been created so far (strk_destroy copes with a half-built context)
    struct Guard {
        strk_ctx *c;
        ~Guard() {
            if (c) strk_destroy(c);
        }
    } guard{ctx};
    ctx->device = device;
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    ctx->n_sm = prop.multiProcessorCount;
    ctx->gap = gap_open;
    ctx->end_flags = end_flags;
    ctx->tie_flags = tie_flags;
    build_lut(ctx->h_consts.lut);
    for (int a = 0; a < STRK_NSYM; ++a)
        for (int b = 0; b < STRK_NSYM; ++b) {
            int v = matrix[a * STRK_NSYM + b];
            if (v < -60 || v > 60) return set_err(STRK_ERR_ARG, "matrix entry %d out of range [-60, 60]", v);
            ctx->h_consts.smat[a * STRK_NSYM + b] = (signed char)v;
        }
    for (int b = 0; b < STRK_NSYM; ++b) {
        ctx->h_consts.smat[STRK_PAD_FREE * STRK_NSYM + b] = 0;
        ctx->h_consts.smat[STRK_PAD_PEN * STRK_NSYM + b] = (signed char)(-2 * gap_open);
    }
    ctx->h_consts.gap = gap_open;
    ctx->h_consts.end_flags = end_flags;
    {
        // PRMT tables of the packed kernel: byte c of t8[b] = score(row class c, column symbol b) + 2g
        static const int class_code[7] = {0, 1, 2, 3, 14, 15, 16};  // A C G T N X other
        int ok = 1;
        for (int b = 0; b < STRK_NSYM; ++b) {
            unsigned long long tf = 0, tb = 0;
            for (int c = 0; c < 7; ++c) {
                int v = matrix[class_code[c] * STRK_NSYM + b] + 2 * gap_open;
                if (v < 0 || v > 127) ok = 0;
                tf |= (unsigned long long)(v & 0xff) << (8 * c);
            }
            tb = tf;  // byte 7 (pad rows) stays 0: pad rows copy the row above them (dp_packed.cuh, borders)
            ctx->h_consts.t8f[b] = tf;
            ctx->h_consts.t8b[b] = tb;
        }
        for (int a = 0; a < STRK_NSYM; ++a)
            for (int b = 0; b < STRK_NSYM; ++b) {
                int v = matrix[a * STRK_NSYM + b] + 2 * gap_open;
                if (v < 0 || v > 127) ok = 0;
            }
        for (int k = 0; k <= STRK_SMAT_ROWS; ++k) ctx->h_consts.cls_of[k] = 0x80;
        for (int c = 0; c < 7; ++c) ctx->h_consts.cls_of[class_code[c]] = (unsigned char)c;
        ctx->h_consts.cls_of[STRK_PAD_FREE] = 7;
        ctx->h_consts.cls_of[STRK_PAD_PEN] = 7;
        for (int k = 0; k <= STRK_SMAT_ROWS; ++k) {
            const unsigned c = ctx->h_consts.cls_of[k];
            unsigned w = 0x800u | 0x88u;  // not representable
            if (!(c & 0x80)) {
                const unsigned cls = c & 7u;
                const unsigned add = cls < 4 || cls == 7 ? 0u : (unsigned)(ctx->h_consts.t8f[0] >> (8 * cls)) & 0xffu;
                w = (cls < 4 ? cls : 8u) | ((cls < 4 ? 4u + cls : 8u) << 4) | (cls << 8) |
                    ((cls < 4 || cls == 7) ? 0u : 0x1000u) | (add << 16);
            }
            ctx->h_consts.rowinfo[k] = w;
        }
        ctx->h_consts.packed_ok = ok;
        int one = 1;  // one-table flank path: a non-ACGT row symbol must score the same against A, C, G and T
        for (int c = 4; c < 7; ++c)
            for (int b = 1; b < 4; ++b)
                if (matrix[class_code[c] * STRK_NSYM + b] != matrix[class_code[c] * STRK_NSYM]) one = 0;
        ctx->h_consts.one_table_ok = one;
        for (int k = 0; k < 32; ++k) ctx->h_consts.one_v[k] = 1u;
    }
    {
        int lo = 0, hi = 0;
        CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));  // lo = least, hi = greatest (numerically smaller)
        ctx->prio_hi = hi;
        CU(cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, hi));
        CU(cudaStreamCreateWithPriority(&ctx->fill_stream, cudaStreamNonBlocking, lo));
    }
    CU(cudaMalloc((void **)&ctx->d_consts, sizeof(ScoreConsts)));
    CU(cudaMemcpyAsync(ctx->d_consts, &ctx->h_consts, sizeof(ScoreConsts), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaMalloc((void **)&ctx->d_queue, (Q_CLASS + STRK_PK_NBIN + 1) * sizeof(unsigned int)));
    CU(cudaMalloc((void **)&ctx->d_acc, 4 * sizeof(double)));
    CU(cudaMalloc((void **)&ctx->d_plan, sizeof(PlanStats)));
    CU(cudaMalloc((void **)&ctx->d_bin_off, STRK_PK_NBIN * sizeof(unsigned int)));
    for (int k = 0; k < 6; ++k) CU(cudaEventCreate(&ctx->ev[k]));
    guard.c = nullptr;
    *out = ctx;
    return STRK_OK;
}

extern "C" int strk_batch_free(strk_ctx *ctx, strk_batch *b);

extern "C" int strk_sync(strk_ctx *ctx) {
    if (!ctx) return set_err(STRK_ERR_ARG, "strk_sync: null context");
    CU(cudaSetDevice(ctx->device));
    for (int k = 0; k < STRK_PK_NBIN; ++k)
        if (ctx->side[k]) CU(cudaStreamSynchronize(ctx->side[k]));
    CU(cudaStreamSynchronize(ctx->fill_stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return STRK_OK;
}

extern "C" int strk_destroy(strk_ctx *ctx) {
    if (!ctx) return STRK_OK;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    if (ctx->reuse) strk_batch_free(ctx, ctx->reuse);
    ctx->reuse = nullptr;
    if (ctx->ref_batch) strk_batch_free(ctx, ctx->ref_batch);
    ctx->ref_batch = nullptr;
    ctx->ref.release();
    ctx->scratch.release();
    ctx->fams.release();
    ctx->table.release();
    ctx->table64.release();
    ctx->list_a.release();
    ctx->list_b.release();
    ctx->list_d.release();
    ctx->list_c.release();
    ctx->fallback.release();
    ctx->pk_scratch.release();
    for (int k = 0; k < 3; ++k) ctx->al_rep[k].release();
    ctx->al_peaks.release();
    for (int k = 0; k < 12; ++k) ctx->al_i[k].release();
    for (int k = 0; k < 4; ++k) ctx->al_d[k].release();
    ctx->al_rb.release();
    ctx->al_doff.release();
    if (ctx->d_consts) cudaFree(ctx->d_consts);
    if (ctx->d_queue) cudaFree(ctx->d_queue);
    if (ctx->d_acc) cudaFree(ctx->d_acc);
    if (ctx->d_plan) cudaFree(ctx->d_plan);
    if (ctx->d_bin_off) cudaFree(ctx->d_bin_off);
    for (int k = 0; k < 6; ++k)
        if (ctx->ev[k]) cudaEventDestroy(ctx->ev[k]);
    for (int k = 0; k < STRK_PK_NBIN; ++k) {
        if (ctx->side[k]) cudaStreamDestroy(ctx->side[k]);
        if (ctx->side_ev[k]) cudaEventDestroy(ctx->side_ev[k]);
    }
    if (ctx->fork_ev) cudaEventDestroy(ctx->fork_ev);
    if (ctx->fill_stream) cudaStreamDestroy(ctx->fill_stream);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return STRK_OK;
}

extern "C" int strk_host_register(void *ptr, uint64_t bytes) {
    if (!ptr || !bytes) return set_err(STRK_ERR_ARG, "strk_host_register: null/empty buffer");
    CU(cudaHostRegister(ptr, bytes, cudaHostRegisterDefault));
    return STRK_OK;
}
extern "C" int strk_host_unregister(void *ptr) {
    if (!ptr) return set_err(STRK_ERR_ARG, "strk_host_unregister: null buffer");
    CU(cudaHostUnregister(ptr));
    return STRK_OK;
}

extern "C" int strk_get_stats(strk_ctx *ctx, double stats[8]) {
    if (!ctx || !stats) return set_err(STRK_ERR_ARG, "strk_get_stats: null argument");
    memcpy(stats, ctx->stats, sizeof(ctx->stats));
    return STRK_OK;
}

// ------------------------------------------------------------------------------------------------
// validation shared by every entry point that takes sequences
// ------------------------------------------------------------------------------------------------
static int validate_reads(const char *who, uint64_t arena_bytes, const uint64_t *seq_off, const int32_t *lens,
                          int64_t n_reads) {
    for (int64_t r = 0; r < n_reads; ++r) {
        const int32_t *L = lens + 3 * r;
        switch (strk_check_read(L[0], L[1], L[2], seq_off[r], arena_bytes)) {
        case PLAN_ERR_NEG_LEN: return set_err(STRK_ERR_ARG, "%s: read %lld has a negative length", who, (long long)r);
        case PLAN_ERR_EMPTY:
            return set_err(STRK_ERR_ARG, "%s: read %lld is empty (fl + tr + fr has no bases)", who, (long long)r);
        case PLAN_ERR_TOO_LONG:
            return set_err(STRK_ERR_ARG, "%s: read %lld is too long (%lld)", who, (long long)r, (long long)L[0] + L[1] + L[2]);
        case PLAN_ERR_PAST_ARENA:
            return set_err(STRK_ERR_ARG, "%s: read %lld runs past the end of the arena", who, (long long)r);
        }
    }
    return STRK_OK;
}

static int validate_motifs(const char *who, uint64_t arena_bytes, const uint64_t *motif_off, const int32_t *motif_len,
                           int64_t n) {
    for (int64_t l = 0; l < n; ++l) {
        switch (strk_check_locus(0, 0, 0, motif_off[l], motif_len[l], arena_bytes)) {  // (motifs only: no reads)
        case PLAN_ERR_MOTIF_EMPTY: return set_err(STRK_ERR_ARG, "%s: motif %lld is empty", who, (long long)l);
        case PLAN_ERR_MOTIF_PAST_ARENA:
            return set_err(STRK_ERR_ARG, "%s: motif %lld runs past the end of the arena", who, (long long)l);
        }
    }
    return STRK_OK;
}

// ------------------------------------------------------------------------------------------------
// general DP launch
// ------------------------------------------------------------------------------------------------
// One family per CTA (dp_general.cuh): the strips of a long read run as a pipeline over the warps of the CTA.
// Throughput shape: GEN_WARPS warps per CTA, 16 / GEN_WARPS CTAs per SM (128 registers per thread).
// Latency shape: a launch that holds long (multi-strip) reads but no more families than fit the SMs at 8 warps each -- a
// locus or a few per call, the widening passes of a block of expansions -- is bound by the time of ONE read; there a
// CTA runs 8 warps, so that twice as many strips of a read are in flight.  Measured on 21 reads of 6 147 rows
// (profiles/r2_general_latency_shape.txt): 2.96 ms at 4 warps, 2.36 ms at 8, 2.52 ms at 16 -- a warp alone on its
// scheduler issues one instruction per 3.7 cycles (dependent issue), and beyond 2 warps per scheduler the strips of one
// read contend for the same issue slots and ALU pipe, so the gain stops at 8.
static int general_latency_warps() {  // (STRK_GEN_LATENCY_WARPS: measurement switch)
    static const int w = getenv("STRK_GEN_LATENCY_WARPS") ? atoi(getenv("STRK_GEN_LATENCY_WARPS")) : 8;
    return std::min(std::max(w, GEN_WARPS), GEN_WARPS_MAX);
}

struct GenShape {
    int grid, warps;
    size_t scratch;  // ints: per CTA [b_len][warps + 1 boundary rows of rowlen]
};

static GenShape general_shape(strk_ctx *ctx, long long n_fams, int b_len, int rowlen, bool latency) {
    GenShape g;
    g.warps = latency ? general_latency_warps() : GEN_WARPS;
    long long blocks = n_fams;
    const long long cap = (long long)ctx->n_sm * (16 / g.warps);  // persistent
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    g.grid = (int)blocks;
    g.scratch = ((size_t)b_len + (size_t)(g.warps + 1) * (size_t)rowlen) * (size_t)g.grid;
    return g;
}

// most families a launch may hold and still take the latency shape (STRK_GEN_LATENCY_MAX: measurement switch)
static long long lat_max(strk_ctx *ctx) {
    static const long long env = getenv("STRK_GEN_LATENCY_MAX") ? atoll(getenv("STRK_GEN_LATENCY_MAX")) : -1;
    return env >= 0 ? env : (long long)ctx->n_sm * (16 / general_latency_warps());  // one wave of latency-shape CTAs
}

static bool general_latency_mode(strk_ctx *ctx, long long n_fams, int rowlen, bool dev_count) {
    static const bool off = getenv("STRK_GEN_LATENCY") && atoi(getenv("STRK_GEN_LATENCY")) == 0;  // (measurement switch)
    return !off && !dev_count && rowlen > 2 && n_fams <= lat_max(ctx);
}

// scratch that any general launch of up to n_fams families may need (either shape)
static size_t general_scratch_max(strk_ctx *ctx, long long n_fams, int b_len, int rowlen) {
    size_t a = general_shape(ctx, n_fams, b_len, rowlen, false).scratch;
    if (rowlen > 2) a = std::max(a, general_shape(ctx, std::min(n_fams, lat_max(ctx)), b_len, rowlen, true).scratch);
    return a;
}

static int launch_general(strk_ctx *ctx, bool ref, const FamDesc *d_fams, const int *d_order, long long n_fams,
                          const unsigned char *d_arena, void *d_table, int b_len, int rowlen, cudaStream_t st,
                          const unsigned int *d_count = nullptr) {
    // d_count != nullptr: the list length lives on the device; n_fams is only its upper bound
    if (n_fams <= 0) return STRK_OK;
    if (d_count && n_fams > (long long)ctx->n_sm * 4) n_fams = (long long)ctx->n_sm * 4;
    if (n_fams > 0x7fffffffLL) return set_err(STRK_ERR_ARG, "too many families in one launch");
    const GenShape gs = general_shape(ctx, n_fams, b_len, rowlen, general_latency_mode(ctx, n_fams, rowlen, d_count != nullptr));
    const int grid = gs.grid, GEN_THREADS = gs.warps * 32;
    const size_t total = gs.scratch;
    if (ctx->scratch.reserve(total) != cudaSuccess) {
        cudaGetLastError();
        return set_err(STRK_ERR_NOMEM, "cannot allocate %zu bytes of DP scratch", total * sizeof(int));
    }
    unsigned int *queue = ctx->counter(Q_GENERAL);
    CU(cudaMemsetAsync(queue, 0, sizeof(unsigned int), st));
    if (ref)
        dp_general_kernel<true><<<grid, GEN_THREADS, 0, st>>>(d_fams, d_order, (int)n_fams, d_arena, ctx->d_consts,
                                                              d_table, ctx->scratch.p, rowlen, b_len, queue, d_count);
    else
        dp_general_kernel<false><<<grid, GEN_THREADS, 0, st>>>(d_fams, d_order, (int)n_fams, d_arena, ctx->d_consts,
                                                               d_table, ctx->scratch.p, rowlen, b_len, queue, d_count);
    CU(cudaGetLastError());
    ctx->stats[2] += 1;
    return STRK_OK;
}

// ------------------------------------------------------------------------------------------------
// packed DP launch (one template instantiation per R; persistent warps, per-warp L2-resident scratch)
// ------------------------------------------------------------------------------------------------
template <int R, int L>
static int launch_packed_r(strk_ctx *ctx, const FamDesc *fams, const int *list, int n, const unsigned char *arena,
                           int *table, PackedDims dims, cudaStream_t st, int ref_mode, size_t *plan_scratch,
                           long long scratch_off) {
    // plan_scratch != nullptr: only report the capture scratch (uint4 units) this launch needs.
    // scratch_off >= 0: the launch uses pk_scratch + scratch_off, reserved by the caller (concurrent class launches).
    constexpr int HALVES = 32 / L;
    const size_t smem = pk_smem_bytes(R, dims, L);
    // the opt-in shared-memory size is a per-device attribute of the function, shared by every context of the
    // process on that device (the streamed path keeps two): only ever raised, under a lock
    {
        static std::mutex mu;
        static size_t configured[64] = {0};
        std::lock_guard<std::mutex> lock(mu);
        size_t &cur = configured[ctx->device & 63];
        if (smem > cur) {
            CU(cudaFuncSetAttribute(dp_packed_kernel<R, L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            cur = smem;
        }
    }
    int per_sm = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, dp_packed_kernel<R, L>, pk_warps(L) * 32, smem));
    if (per_sm < 1) return set_err(STRK_ERR_CUDA, "packed kernel R=%d L=%d does not fit an SM (%zu B shared)", R, L, smem);
    long long grid = (long long)per_sm * ctx->n_sm;
    const long long need = ((long long)n + pk_warps(L) * HALVES - 1) / (pk_warps(L) * HALVES);
    if (grid > need) grid = need;
    const size_t words = pk_scratch_words_per_unit(R, dims.w_max, L) * (size_t)grid * pk_warps(L) * HALVES;
    if (plan_scratch) {
        *plan_scratch = (words + 3) / 4;
        return STRK_OK;
    }
    if (scratch_off < 0 && ctx->pk_scratch.reserve((words + 3) / 4) != cudaSuccess) {
        cudaGetLastError();
        return set_err(STRK_ERR_NOMEM, "cannot allocate %zu bytes of capture scratch", words * 4);
    }
    // The capture scratch is written and read back within one read's lifetime and then overwritten by the next read of
    // the same warp.  Keeping it resident in L2 (persisting access window) was measured: 1176 -> 89 MB of DRAM traffic
    // per launch of the R = 10 class, no change in kernel time (the kernel is integer-issue bound, the write-backs use
    // ~10 % of HBM bandwidth), -2 % on the streamed path where two contexts' windows compete for the set-aside: it is
    // not pinned (DESIGN.md 5.1).
    unsigned int *work_counter = ctx->counter(Q_CLASS + (L == 16 ? R / 2 : R));  // one queue per rows-per-lane class
    CU(cudaMemsetAsync(work_counter, 0, sizeof(unsigned int), st));
    dp_packed_kernel<R, L><<<(unsigned)grid, pk_warps(L) * 32, smem, st>>>(fams, list, n, arena, ctx->d_consts, table, dims,
                                                                        ctx->pk_scratch.p + (scratch_off > 0 ? scratch_off : 0),
                                                                        ctx->fallback.p, ctx->counter(Q_FALLBACK), ref_mode,
                                                                        work_counter);
    CU(cudaGetLastError());
    ctx->stats[2] += 1;
    return STRK_OK;
}

// Lanes per read of a rows-per-lane class: reads of the classes up to PK_PAIR_RMAX (db < 32 * PK_PAIR_RMAX bases) are
// swept two per warp, 16 lanes x 2R rows each (half the skew, half the per-step overhead per read).
// Larger classes were measured slower paired (R = 9: -1.2 %, 10: -1.8 %, 12: -3.2 %: 2R rows per lane need 127+
// registers).  STRK_PK_PAIRS=<largest paired class, 0 = none, at most 8> overrides the default (measurement only).
#define PK_PAIR_RMAX 8
static int pk_lanes_for_class(int R) {
    static const int rmax = [] {
        const char *e = getenv("STRK_PK_PAIRS");
        const int v = e ? atoi(e) : PK_PAIR_RMAX;
        return v < 0 ? 0 : (v > PK_PAIR_RMAX ? PK_PAIR_RMAX : v);
    }();
    return R <= rmax ? 16 : 32;
}
// sizes of the class' shared-memory tables for the lane count it runs with
static PackedDims pk_dims_for_class(int R, int max_flank, int max_m, int w_max) {
    const int L = pk_lanes_for_class(R);
    PackedDims d;
    d.colt_entries = max_flank + 2 * L;  // columns -(L - 1) .. flank + (L - 1), one spare
    d.prof_words = L == 16 ? pk_prof_words(2 * R, max_m, 16) : pk_prof_words(R, max_m, 32);
    d.w_max = w_max;
    return d;
}
static size_t pk_smem_for_class(int R, const PackedDims &d) {
    return pk_lanes_for_class(R) == 16 ? pk_smem_bytes(2 * R, d, 16) : pk_smem_bytes(R, d, 32);
}

// ref_mode: the families are reference windows and `table` holds the 64-bit boundary keys (score_ref_boundaries)
static int launch_packed(strk_ctx *ctx, int R, const FamDesc *fams, const int *list, int n, const unsigned char *arena,
                         int *table, PackedDims dims, cudaStream_t st, int ref_mode = 0, size_t *plan_scratch = nullptr,
                         long long scratch_off = -1) {
    if (pk_lanes_for_class(R) == 16) {
        switch (R) {
#define PK_CASE(N) \
    case N: return launch_packed_r<2 * N, 16>(ctx, fams, list, n, arena, table, dims, st, ref_mode, plan_scratch, scratch_off);
            PK_CASE(2) PK_CASE(3) PK_CASE(4) PK_CASE(5) PK_CASE(6) PK_CASE(7) PK_CASE(8)
#undef PK_CASE
            default: break;
        }
    }
    switch (R) {
#define PK_CASE(N) \
    case N: return launch_packed_r<N, 32>(ctx, fams, list, n, arena, table, dims, st, ref_mode, plan_scratch, scratch_off);
        PK_CASE(2) PK_CASE(3) PK_CASE(4) PK_CASE(5) PK_CASE(6) PK_CASE(7) PK_CASE(8) PK_CASE(9) PK_CASE(10) PK_CASE(11)
        PK_CASE(12) PK_CASE(13) PK_CASE(14) PK_CASE(15) PK_CASE(16)
#undef PK_CASE
        default: return set_err(STRK_ERR_ARG, "packed kernel: no instantiation for %d rows per lane", R);
    }
}

// Whether the packed kernel takes a pass of windows of W sizes (a reference window, a forward and a reverse column per
// size, counts twice), and a family's class in such a pass.  The planners gate on the matrix only: a batch's windows are
// decided per pass.
static bool pk_window_ok(const strk_ctx *ctx, int kernel, int ref_mode, int W) {
    return kernel != STRK_KERNEL_GENERAL && ctx->h_consts.packed_ok && (ref_mode ? 2 * W : W) <= PK_WINDOW_MAX;
}
static int pk_class(const strk_ctx *ctx, int kernel, int ref_mode, int W, int fl, int tr, int fr, int m) {
    return pk_window_ok(ctx, kernel, ref_mode, W) ? strk_pk_class(fl, tr, fr, m) : 0;
}

// Table width (PackedDims::w_max) of a packed class whose widest window holds W sizes
static int pk_table_w(int ref_mode, int W) { return ref_mode ? 2 * W - 1 : (W + 3) / 4 * 4; }

// One DP pass: list[0] through the general kernel, list[k >= 1] through the packed kernel (or, when the class' tables do
// not fit shared memory, the general kernel), then the packed kernel's fallbacks (a device-side list, Q_FALLBACK long)
// through the general kernel; *n_packed = the items the packed launches took.  A pass without packed items is one
// general launch.  The general launch of list[0] is a handful of families (reads / reference windows of 512+ bases,
// IUPAC reads) whose duration is the LATENCY of one family's chain (0.3 - 0.6 ms) whatever the grid: it starts first, on
// its own side stream, under the packed launches (it used to be 3 % of a 32 768-locus read step).  Large passes run the
// classes back to back on `st` (several streams were measured slower there, -2.8 %: concurrent grids with different
// footprints fragment the SMs); small passes, where each launch lasts one read's sweep whatever its grid, run every
// class on its own side stream with its own slice of the capture scratch, so the launches overlap.
// strk_ref_counts queues several passes before it synchronises, so no reservation here may reallocate a buffer that a
// queued pass still reads: it reserves the fallback list (and its class lists) for the whole call up front.
static int launch_pass(strk_ctx *ctx, const DpPass &p, cudaStream_t st, long long *n_packed) {
    static const long long fan_max = [] {
        const char *e = getenv("STRK_PK_FANOUT_MAX");  // reads per pass up to which the classes overlap
        return e ? atoll(e) : 131072LL;
    }();
    const bool ref = p.ref_mode != 0;
    *n_packed = 0;
    long long packed_total = 0;
    for (int k = 1; k < STRK_PK_NBIN; ++k) packed_total += p.cnt[k];
    if (!packed_total) return launch_general(ctx, ref, p.fams, p.list[0], p.cnt[0], p.arena, p.table, p.b_len, p.rowlen, st);

    PackedDims dims[STRK_PK_NBIN];
    bool fits[STRK_PK_NBIN] = {false};
    bool overlap = p.cnt[0] > 0;  // (not when a class runs on the general kernel itself)
    long long fams_max = std::max(p.cnt[0], std::min(packed_total, (long long)ctx->n_sm * 4));
    for (int k = 1; k < STRK_PK_NBIN; ++k) {
        if (!p.cnt[k]) continue;
        dims[k] = pk_dims_for_class(k, p.flank[k], p.mmax[k], pk_table_w(p.ref_mode, p.w[k]));
        fits[k] = pk_smem_for_class(k, dims[k]) <= 200 * 1024;
        overlap = overlap && fits[k];
        fams_max = std::max(fams_max, p.cnt[k]);
    }
    // scratch of the largest general launch of this pass, reserved before anything is in flight
    const size_t total = general_scratch_max(ctx, fams_max, p.b_len, p.rowlen);
    if (ctx->scratch.reserve(total) != cudaSuccess) {
        cudaGetLastError();
        return set_err(STRK_ERR_NOMEM, "cannot allocate %zu bytes of DP scratch", total * sizeof(int));
    }
    if (ctx->fallback.reserve((size_t)packed_total) != cudaSuccess) {
        cudaGetLastError();
        return set_err(STRK_ERR_NOMEM, "cannot allocate the fallback list");
    }
    CU(cudaMemsetAsync(ctx->counter(Q_FALLBACK), 0, sizeof(unsigned int), st));
    if (!ctx->fork_ev) CU(cudaEventCreateWithFlags(&ctx->fork_ev, cudaEventDisableTiming));
    int rc = STRK_OK;
    if (overlap) {
        if (!ctx->side[0]) CU(cudaStreamCreateWithPriority(&ctx->side[0], cudaStreamNonBlocking, ctx->prio_hi));
        if (!ctx->side_ev[0]) CU(cudaEventCreateWithFlags(&ctx->side_ev[0], cudaEventDisableTiming));
        CU(cudaEventRecord(ctx->fork_ev, st));
        CU(cudaStreamWaitEvent(ctx->side[0], ctx->fork_ev, 0));
        rc = launch_general(ctx, ref, p.fams, p.list[0], p.cnt[0], p.arena, p.table, p.b_len, p.rowlen, ctx->side[0]);
        if (rc) return rc;
        CU(cudaEventRecord(ctx->side_ev[0], ctx->side[0]));
    }
    long long fan_off[STRK_PK_NBIN];
    bool fan_out = false;
    if (p.n_slots <= fan_max) {
        size_t scratch = 0;
        int n_classes = 0;
        for (int k = STRK_PK_RMAX; k >= 1; --k) {
            if (!p.cnt[k] || !fits[k]) continue;
            size_t need = 0;
            rc = launch_packed(ctx, k, p.fams, p.list[k], (int)p.cnt[k], p.arena, (int *)p.table, dims[k], st, p.ref_mode,
                               &need);
            if (rc) return rc;
            fan_off[k] = (long long)scratch;
            scratch += need;
            ++n_classes;
        }
        if (n_classes >= 2) {
            if (ctx->pk_scratch.reserve(scratch) != cudaSuccess) {
                cudaGetLastError();
                return set_err(STRK_ERR_NOMEM, "cannot allocate %zu bytes of capture scratch", scratch * sizeof(uint4));
            }
            CU(cudaEventRecord(ctx->fork_ev, st));
            fan_out = true;
        }
    }
    for (int k = STRK_PK_RMAX; k >= 1; --k) {
        if (!p.cnt[k]) continue;
        if (!fits[k]) {
            rc = launch_general(ctx, ref, p.fams, p.list[k], p.cnt[k], p.arena, p.table, p.b_len, p.rowlen, st);
            if (rc) return rc;
            continue;
        }
        if (fan_out) {
            if (!ctx->side[k]) CU(cudaStreamCreateWithPriority(&ctx->side[k], cudaStreamNonBlocking, ctx->prio_hi));
            if (!ctx->side_ev[k]) CU(cudaEventCreateWithFlags(&ctx->side_ev[k], cudaEventDisableTiming));
            CU(cudaStreamWaitEvent(ctx->side[k], ctx->fork_ev, 0));
            rc = launch_packed(ctx, k, p.fams, p.list[k], (int)p.cnt[k], p.arena, (int *)p.table, dims[k], ctx->side[k],
                               p.ref_mode, nullptr, fan_off[k]);
            if (rc) return rc;
            CU(cudaEventRecord(ctx->side_ev[k], ctx->side[k]));
            CU(cudaStreamWaitEvent(st, ctx->side_ev[k], 0));
        } else {
            rc = launch_packed(ctx, k, p.fams, p.list[k], (int)p.cnt[k], p.arena, (int *)p.table, dims[k], st, p.ref_mode);
            if (rc) return rc;
        }
        *n_packed += p.cnt[k];
    }
    if (overlap) {
        CU(cudaStreamWaitEvent(st, ctx->side_ev[0], 0));
    } else {
        rc = launch_general(ctx, ref, p.fams, p.list[0], p.cnt[0], p.arena, p.table, p.b_len, p.rowlen, st);
        if (rc) return rc;
    }
    if (*n_packed)
        return launch_general(ctx, ref, p.fams, ctx->fallback.p, *n_packed, p.arena, p.table, p.b_len, p.rowlen, st,
                              ctx->counter(Q_FALLBACK));
    return STRK_OK;
}

// ------------------------------------------------------------------------------------------------
// batches
// ------------------------------------------------------------------------------------------------
// Reserves the per-read and per-locus buffers of `b` for n_reads reads of n_loci loci, points the d_* aliases at them
// and clears the work plan (batch_plan / batch_plan_host fill it in).  The arena is the caller's to set.
static cudaError_t batch_bind(strk_batch *b, long long n_reads, long long n_loci) {
    const size_t nr = (size_t)(n_reads ? n_reads : 1), nl = (size_t)(n_loci ? n_loci : 1);
    cudaError_t e = b->seq_off.reserve(nr);
    if (e == cudaSuccess) e = b->lens.reserve(3 * nr);
    if (e == cudaSuccess) e = b->est.reserve(nr);
    if (e == cudaSuccess) e = b->read_locus.reserve(nr);
    if (e == cudaSuccess) e = b->order.reserve(nr);
    if (e == cudaSuccess) e = b->bin.reserve(nr);
    if (e == cudaSuccess) e = b->out.reserve(4 * nr);
    if (e == cudaSuccess) e = b->read_begin.reserve((size_t)n_loci + 1);
    if (e == cudaSuccess) e = b->motif_off.reserve(nl);
    if (e == cudaSuccess) e = b->motif_len.reserve(nl);
    if (e == cudaSuccess) e = b->status.reserve(nl);
    b->n_reads = n_reads;
    b->n_loci = n_loci;
    b->d_seq_off = b->seq_off.p, b->d_lens = b->lens.p, b->d_est = b->est.p, b->d_read_locus = b->read_locus.p;
    b->d_order = b->order.p, b->d_out = b->out.p, b->d_read_begin = b->read_begin.p;
    b->d_motif_off = b->motif_off.p, b->d_motif_len = b->motif_len.p, b->d_status = b->status.p;
    b->n_general = 0;
    for (int k = 0; k < STRK_PK_NBIN; ++k) b->bin_off[k] = b->bin_cnt[k] = 0, b->bin_mmax[k] = b->bin_flank[k] = 0;
    b->ext = GenExtent{};
    return e;
}

extern "C" int strk_batch_free(strk_ctx *ctx, strk_batch *b) {
    if (!b) return STRK_OK;
    if (ctx) cudaSetDevice(ctx->device);
    b->release();
    delete b;
    return STRK_OK;
}

// The error of a batch whose planning found one: the first faulty read or locus and its PlanError
static int plan_error(long long index, int kind) {
    static const char *what[] = {"", "has a negative length", "is empty (fl + tr + fr has no bases)", "is too long",
                                 "runs past the end of the arena", "has an out-of-range est_cn", "has an empty motif",
                                 "has a motif that runs past the end of the arena", "has a non-monotone read_begin"};
    return set_err(STRK_ERR_ARG, "batch: %s %lld %s", kind >= PLAN_ERR_MOTIF_EMPTY ? "locus" : "read", index,
                   what[kind <= 8 ? kind : 0]);
}

// The work plan of a batch from its per-class read counts, per-class maxima and general-kernel extents: segment
// offsets with the general kernel's reads first, then packed classes from R = 16 down to 2 (class 1 stays empty).
static void batch_layout(strk_batch *b, const unsigned *cnt, const int *mmax, const int *flank, const GenExtent &ext) {
    long long acc = cnt[0];
    b->n_general = cnt[0];
    for (int k = STRK_PK_RMAX; k >= 1; --k) {
        b->bin_off[k] = acc;
        b->bin_cnt[k] = cnt[k];
        b->bin_mmax[k] = mmax[k];
        b->bin_flank[k] = flank[k];
        acc += cnt[k];
    }
    b->ext = ext;
}

// Validation + work planning of a batch whose arrays are already on the device (b->d_*, n_reads, n_loci set).
static int batch_plan(strk_ctx *ctx, strk_batch *b, uint64_t arena_bytes) {
    const long long n_reads = b->n_reads, n_loci = b->n_loci;
    cudaStream_t st = ctx->fill_stream;  // (callers hand over host-synchronised data; every path below ends synchronised)
    b->d_rep = nullptr;
    b->n_dup = 0;
    if (n_reads == 0) {
        CU(cudaStreamSynchronize(st));
        return STRK_OK;
    }
    // ---- plan on the device
    PlanStats hp;
    CU(cudaMemsetAsync(ctx->d_plan, 0, sizeof(PlanStats), st));
    CU(cudaMemsetAsync(&ctx->d_plan->first_error, 0xff, sizeof(unsigned long long), st));
    const int T = 256;
    plan_loci_kernel<<<(unsigned)((n_loci + T - 1) / T), T, 0, st>>>(b->d_read_begin, n_loci, n_reads, b->d_motif_off,
                                                                     b->d_motif_len, arena_bytes, b->d_read_locus,
                                                                     ctx->d_plan);
    CU(cudaGetLastError());
    // the read scan dereferences read_locus / motif_len: stop here if the locus table itself is broken
    CU(cudaMemcpyAsync(&hp, ctx->d_plan, sizeof(PlanStats), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (hp.first_error == ~0ull) {
        plan_reads_scan_kernel<<<(unsigned)((n_reads + T - 1) / T), T, 0, st>>>(
            b->d_seq_off, b->d_lens, b->d_est, b->d_read_locus, b->d_motif_len, n_reads, arena_bytes,
            ctx->h_consts.packed_ok, b->bin.p, ctx->d_plan);
        CU(cudaGetLastError());
        // identical reads of a locus share one table (STRK_DEDUPE=0 switches it off: measurement only)
        const char *dd = getenv("STRK_DEDUPE");
        if ((!dd || atoi(dd) != 0) && n_reads > n_loci) {
            if (b->hash.reserve((size_t)n_reads) != cudaSuccess || b->rep.reserve((size_t)n_reads) != cudaSuccess) {
                cudaGetLastError();
                return set_err(STRK_ERR_NOMEM, "batch: cannot allocate the duplicate-read map");
            }
            hash_reads_kernel<<<(unsigned)((n_reads * 32 + T - 1) / T), T, 0, st>>>(b->d_arena, b->d_seq_off, b->d_lens, b->d_est,
                                                                                 n_reads, ctx->d_plan, b->hash.p);
            CU(cudaGetLastError());
            dedupe_loci_kernel<<<(unsigned)((n_loci * 32 + T - 1) / T), T, 0, st>>>(b->d_arena, b->d_seq_off, b->d_lens, b->d_est,
                                                                                  b->d_read_begin, n_loci, b->hash.p, b->bin.p,
                                                                                  ctx->d_plan, b->rep.p);
            CU(cudaGetLastError());
            b->d_rep = b->rep.p;
        }
        CU(cudaMemcpyAsync(&hp, ctx->d_plan, sizeof(PlanStats), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    if (hp.first_error != ~0ull) return plan_error((long long)(hp.first_error >> 8), (int)(hp.first_error & 0xff));
    batch_layout(b, hp.bin_cnt, hp.bin_mmax, hp.bin_flank, hp.ext);
    b->n_dup = b->d_rep ? (long long)hp.n_dup : 0;
    unsigned off[STRK_PK_NBIN];
    for (int k = 0; k < STRK_PK_NBIN; ++k) off[k] = (unsigned)b->bin_off[k];
    CU(cudaMemcpyAsync(ctx->d_bin_off, off, sizeof(off), cudaMemcpyHostToDevice, st));
    plan_reads_scatter_kernel<<<(unsigned)((n_reads + T - 1) / T), T, 0, st>>>(b->bin.p, n_reads, ctx->d_bin_off,
                                                                              ctx->d_plan, b->d_order, b->d_rep);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(st));  // `off` is on this stack frame; the caller's buffers may go away after return
    return STRK_OK;
}

// The same validation + planning on the host, for small batches (the per-call wrappers of the drop-in API send one
// read at a time): no planning kernels, no read-backs, one stream synchronisation.  Loci are checked before reads,
// and the first fault is reported, as on the device.
#define STRK_SMALL_BATCH 512
static int batch_plan_host(strk_ctx *ctx, strk_batch *b, uint64_t arena_bytes, const uint64_t *seq_off, const int32_t *lens,
                           const int32_t *est_cn, const int64_t *read_begin, const uint64_t *motif_off,
                           const int32_t *motif_len) {
    const long long n_reads = b->n_reads, n_loci = b->n_loci;
    cudaStream_t st = ctx->fill_stream;
    b->d_rep = nullptr;  // small batches: every read gets its own table
    b->n_dup = 0;
    if (n_reads == 0) {
        CU(cudaStreamSynchronize(st));
        return STRK_OK;
    }
    std::vector<int> read_locus((size_t)n_reads, 0), order((size_t)n_reads);
    std::vector<unsigned char> bin((size_t)n_reads, 0);
    for (long long l = 0; l < n_loci; ++l) {
        const long long r0 = read_begin[l], r1 = read_begin[l + 1];
        const int kind = strk_check_locus(r0, r1, n_reads, motif_off[l], motif_len[l], arena_bytes);
        if (kind) return plan_error(l, kind);
        for (long long r = r0; r < r1; ++r) read_locus[(size_t)r] = (int)l;
    }
    unsigned cnt[STRK_PK_NBIN] = {0};
    int mmax[STRK_PK_NBIN] = {0}, flank[STRK_PK_NBIN] = {0};
    GenExtent ext = {};
    for (long long r = 0; r < n_reads; ++r) {
        const int fl = lens[3 * r], tr = lens[3 * r + 1], fr = lens[3 * r + 2];
        const int m = motif_len[read_locus[(size_t)r]], est = est_cn[r];
        int kind = strk_check_read(fl, tr, fr, seq_off[r], arena_bytes);
        if (!kind) kind = strk_check_est(est, m);
        if (kind) return plan_error(r, kind);
        const int bb = ctx->h_consts.packed_ok ? strk_pk_class(fl, tr, fr, m) : 0;
        if (bb) {
            mmax[bb] = std::max(mmax[bb], m);
            flank[bb] = std::max(flank[bb], std::max(fl, fr));
        }
        ext.add(fl, fr, fl + tr + fr, m, est);
        bin[(size_t)r] = (unsigned char)bb;
        ++cnt[bb];
    }
    batch_layout(b, cnt, mmax, flank, ext);
    long long off[STRK_PK_NBIN];
    std::copy(b->bin_off, b->bin_off + STRK_PK_NBIN, off);
    for (long long r = 0; r < n_reads; ++r) order[(size_t)off[bin[(size_t)r]]++] = (int)r;
    CU(cudaMemcpyAsync(b->d_read_locus, read_locus.data(), (size_t)n_reads * sizeof(int), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(b->d_order, order.data(), (size_t)n_reads * sizeof(int), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(b->bin.p, bin.data(), (size_t)n_reads, cudaMemcpyHostToDevice, st));
    // The caller's arrays (possibly pinned: truly asynchronous DMA) and the vectors above are still being read by the
    // copies queued on `st`; the header promises that no host pointer is kept after a call returns, and strk_batch_run
    // may run on a caller stream that is not ordered after `st`.
    CU(cudaStreamSynchronize(st));
    return STRK_OK;
}

// H2D into (possibly recycled) device buffers, then validation + work planning on the device (plan.cuh)
static int batch_fill(strk_ctx *ctx, strk_batch *b, const uint8_t *arena, uint64_t arena_bytes, const uint64_t *seq_off,
                      const int32_t *lens, const int32_t *est_cn, int64_t n_reads, const int64_t *read_begin,
                      const uint64_t *motif_off, const int32_t *motif_len, int64_t n_loci,
                      int arena_format = STRK_ARENA_ASCII) {
    if (arena_format != STRK_ARENA_ASCII && arena_format != STRK_ARENA_NIBBLE)
        return set_err(STRK_ERR_ARG, "batch: unknown arena format %d", arena_format);
    if (n_reads < 0 || n_loci < 0 || n_reads > 0x7ffffff0LL || n_loci > 0x7ffffff0LL)
        return set_err(STRK_ERR_ARG, "batch: bad counts (%lld reads, %lld loci)", (long long)n_reads, (long long)n_loci);
    if ((n_reads && (!arena || !seq_off || !lens || !est_cn)) || !read_begin || (n_loci && (!motif_off || !motif_len)))
        return set_err(STRK_ERR_ARG, "batch: null array");
    if (read_begin[0] != 0 || read_begin[n_loci] != n_reads)
        return set_err(STRK_ERR_ARG, "batch: read_begin must run from 0 to n_reads");
    CU(cudaSetDevice(ctx->device));
    b->h_read_begin.assign(read_begin, read_begin + n_loci + 1);

    cudaStream_t st = ctx->fill_stream;
    cudaError_t e = batch_bind(b, n_reads, n_loci);
#define UP(dst, src, n) \
    if (e == cudaSuccess && (n)) e = cudaMemcpyAsync(b->dst, src, (size_t)(n) * sizeof(*b->dst), cudaMemcpyHostToDevice, st)
    if (arena_format == STRK_ARENA_NIBBLE) {
        // packed bytes in, byte-per-symbol arena out (offsets and lengths are in symbols either way)
        const size_t quads = (size_t)((arena_bytes + 15) / 16);
        if (e == cudaSuccess) e = b->arena4.reserve(quads ? quads : 1);
        if (e == cudaSuccess) e = b->arena.reserve((size_t)(arena_bytes ? 2 * arena_bytes : 1));
        b->d_arena = b->arena.p;
        if (e == cudaSuccess && arena_bytes) {
            e = cudaMemcpyAsync(b->arena4.p, arena, (size_t)arena_bytes, cudaMemcpyHostToDevice, st);
            const unsigned long long threads = (arena_bytes >> 4) + 1;
            if (e == cudaSuccess) {
                expand_nibbles_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(b->arena4.p, arena_bytes, b->arena.p);
                e = cudaGetLastError();
            }
        }
        arena_bytes *= 2;  // symbols
    } else {
        if (e == cudaSuccess) e = b->arena.reserve((size_t)(arena_bytes ? arena_bytes : 1));
        b->d_arena = b->arena.p;
        UP(d_arena, arena, arena_bytes);
    }
    UP(d_seq_off, seq_off, n_reads);
    UP(d_lens, lens, 3 * n_reads);
    UP(d_est, est_cn, n_reads);
    UP(d_read_begin, read_begin, n_loci + 1);
    UP(d_motif_off, motif_off, n_loci);
    UP(d_motif_len, motif_len, n_loci);
#undef UP
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(e == cudaErrorMemoryAllocation ? STRK_ERR_NOMEM : STRK_ERR_CUDA, "batch upload: %s",
                       cudaGetErrorString(e));
    }
    if (n_reads <= STRK_SMALL_BATCH) return batch_plan_host(ctx, b, arena_bytes, seq_off, lens, est_cn, read_begin, motif_off, motif_len);
    return batch_plan(ctx, b, arena_bytes);
}

extern "C" int strk_batch_create(strk_ctx *ctx, strk_batch **out) {
    if (!ctx || !out) return set_err(STRK_ERR_ARG, "strk_batch_create: null context/output");
    *out = new (std::nothrow) strk_batch();
    if (!*out) return set_err(STRK_ERR_NOMEM, "out of host memory");
    return STRK_OK;
}

extern "C" int strk_batch_fill(strk_ctx *ctx, strk_batch *b, const uint8_t *arena, uint64_t arena_bytes,
                               const uint64_t *seq_off, const int32_t *lens, const int32_t *est_cn, int64_t n_reads,
                               const int64_t *read_begin, const uint64_t *motif_off, const int32_t *motif_len,
                               int64_t n_loci) {
    if (!ctx || !b) return set_err(STRK_ERR_ARG, "strk_batch_fill: null context/batch");
    return batch_fill(ctx, b, arena, arena_bytes, seq_off, lens, est_cn, n_reads, read_begin, motif_off, motif_len, n_loci);
}

extern "C" int strk_batch_fill_fmt(strk_ctx *ctx, strk_batch *b, int arena_format, const uint8_t *arena,
                                   uint64_t arena_bytes, const uint64_t *seq_off, const int32_t *lens,
                                   const int32_t *est_cn, int64_t n_reads, const int64_t *read_begin,
                                   const uint64_t *motif_off, const int32_t *motif_len, int64_t n_loci) {
    if (!ctx || !b) return set_err(STRK_ERR_ARG, "strk_batch_fill_fmt: null context/batch");
    return batch_fill(ctx, b, arena, arena_bytes, seq_off, lens, est_cn, n_reads, read_begin, motif_off, motif_len, n_loci,
                      arena_format);
}

extern "C" int strk_batch_upload(strk_ctx *ctx, const uint8_t *arena, uint64_t arena_bytes, const uint64_t *seq_off,
                                 const int32_t *lens, const int32_t *est_cn, int64_t n_reads, const int64_t *read_begin,
                                 const uint64_t *motif_off, const int32_t *motif_len, int64_t n_loci,
                                 strk_batch **out) {
    if (!ctx || !out) return set_err(STRK_ERR_ARG, "strk_batch_upload: null context/output");
    *out = nullptr;
    strk_batch *b = new (std::nothrow) strk_batch();
    if (!b) return set_err(STRK_ERR_NOMEM, "out of host memory");
    int rc = batch_fill(ctx, b, arena, arena_bytes, seq_off, lens, est_cn, n_reads, read_begin, motif_off, motif_len,
                        n_loci);
    if (rc) {
        strk_batch_free(ctx, b);
        return rc;
    }
    *out = b;
    return STRK_OK;
}

// Replay of a pass over ctx->table (W sizes per slot), one thread per locus of `b` or of d_locus_ids; narrow windows
// take the kernel that keeps each read's row in shared memory.  The caller counts the launch.
static int launch_replay(strk_ctx *ctx, const strk_batch *b, int W, int wd, int ws, const int *d_locus_ids,
                         const long long *d_slot_begin, long long n_list, int max_iters, int range, int step,
                         const int *d_rep, double *d_hint, cudaStream_t st) {
    const auto kernel = W <= REPLAY_WMAX ? replay_reads_small_kernel : replay_reads_kernel;
    kernel<<<(unsigned)((n_list + REPLAY_THREADS - 1) / REPLAY_THREADS), REPLAY_THREADS, 0, st>>>(
        ctx->table.p, W, wd, ws, d_locus_ids, d_slot_begin, (int)n_list, b->d_read_begin, b->d_est, b->d_lens,
        b->d_motif_len, max_iters, range, step, ctx->tie_flags, b->d_out, b->d_status, ctx->counter(Q_MISS), ctx->d_acc,
        d_rep, d_hint);
    CU(cudaGetLastError());
    return STRK_OK;
}

// The classes of a widening pass over the reads of h_read_ids (slot sl = read h_read_ids[sl]): each read in the class
// planned for it at upload time (h_bin, read back once per run), with the batch's class maxima.
static int widening_pass(strk_ctx *ctx, const strk_batch *b, const std::vector<int> &h_read_ids,
                         std::vector<unsigned char> &h_bin, int W, cudaStream_t st, DpPass &p) {
    if (h_bin.empty()) {
        h_bin.resize((size_t)b->n_reads);
        CU(cudaMemcpyAsync(h_bin.data(), b->bin.p, (size_t)b->n_reads, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    ClassLists lists;
    for (int k = 0; k < STRK_PK_NBIN; ++k) lists.flank[k] = b->bin_flank[k], lists.mmax[k] = b->bin_mmax[k], lists.w_max[k] = W;
    // A small pass is launch-latency bound (one read's sweep is ~100 us whatever the grid): its reads run in the largest
    // class of their lane group (pad rows cost nothing there), two launches instead of 15.
    int merged[STRK_PK_NBIN];
    for (int k = 0; k < STRK_PK_NBIN; ++k) merged[k] = k;
    if (h_read_ids.size() <= 8192) {
        bool used[STRK_PK_NBIN] = {false};
        for (int r : h_read_ids) used[h_bin[(size_t)r]] = true;
        for (int L = 16; L <= 32; L += 16) {
            int top = 0;
            for (int k = 1; k < STRK_PK_NBIN; ++k)
                if (used[k] && pk_lanes_for_class(k) == L) top = k;
            for (int k = 1; k < top; ++k)
                if (used[k] && pk_lanes_for_class(k) == L) {
                    merged[k] = top;
                    lists.flank[top] = std::max(lists.flank[top], lists.flank[k]);
                    lists.mmax[top] = std::max(lists.mmax[top], lists.mmax[k]);
                }
        }
    }
    for (size_t sl = 0; sl < h_read_ids.size(); ++sl) lists.add(merged[h_bin[(size_t)h_read_ids[sl]]], (int)sl);
    const int rc = lists.upload(ctx->list_d, st, p);
    if (rc) return rc;
    CU(cudaStreamSynchronize(st));  // `lists` is read by the copy
    return STRK_OK;
}

// The loci of the next widening pass: those of the last pass (pass 0: every locus) whose search left its window
// (status 1; status 2 is an error), their reads as the slots of the pass and each locus' first slot, uploaded to
// ctx->list_a (reads), list_b (loci) and list_c (first slots).
static int next_loci(strk_ctx *ctx, const strk_batch *b, bool from_pass0, int max_iters, std::vector<int> &h_locus_ids,
                     std::vector<int> &h_read_ids, std::vector<long long> &h_slot_begin, cudaStream_t st) {
    std::vector<unsigned char> h_status((size_t)b->n_loci);
    CU(cudaMemcpy(h_status.data(), b->d_status, (size_t)b->n_loci, cudaMemcpyDeviceToHost));
    std::vector<int> loci;
    h_read_ids.clear();
    h_slot_begin.clear();
    const long long n_last = from_pass0 ? b->n_loci : (long long)h_locus_ids.size();
    for (long long i = 0; i < n_last; ++i) {
        const int l = from_pass0 ? (int)i : h_locus_ids[(size_t)i];
        if (!h_status[(size_t)l]) continue;
        if (h_status[(size_t)l] == 2)
            return set_err(STRK_ERR_SEARCH, "locus %d: the search scored no size (max_iters = %d)", l, max_iters);
        loci.push_back(l);
        h_slot_begin.push_back((long long)h_read_ids.size());
        for (long long r = b->h_read_begin[(size_t)l]; r < b->h_read_begin[(size_t)l + 1]; ++r)
            h_read_ids.push_back((int)r);
    }
    h_locus_ids.swap(loci);
    if (ctx->list_a.reserve(h_read_ids.size()) != cudaSuccess || ctx->list_b.reserve(h_locus_ids.size()) != cudaSuccess ||
        ctx->list_c.reserve(h_slot_begin.size()) != cudaSuccess) {
        cudaGetLastError();
        return set_err(STRK_ERR_NOMEM, "cannot allocate widening lists");
    }
    CU(cudaMemcpyAsync(ctx->list_a.p, h_read_ids.data(), h_read_ids.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ctx->list_b.p, h_locus_ids.data(), h_locus_ids.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ctx->list_c.p, h_slot_begin.data(), h_slot_begin.size() * sizeof(long long), cudaMemcpyHostToDevice,
                       st));
    CU(cudaStreamSynchronize(st));
    return STRK_OK;
}

extern "C" int strk_batch_run(strk_ctx *ctx, strk_batch *b, int max_iters, int local_search_range, int step_size,
                              int kernel, void *stream) {
    if (!ctx || !b) return set_err(STRK_ERR_ARG, "strk_batch_run: null argument");
    if (max_iters < 0 || local_search_range < 0 || step_size < 0 || local_search_range > 1000 || step_size > 1000)
        return set_err(STRK_ERR_ARG, "strk_batch_run: bad search parameters");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
    for (int k = 0; k < 8; ++k) ctx->stats[k] = 0;
    if (b->n_reads == 0) {
        return STRK_OK;
    }
    CU(cudaMemsetAsync(ctx->d_acc, 0, 4 * sizeof(double), st));

    // first-pass window half-width around the per-read estimate: the replay of a well-started search visits
    // start +- (range + step); the margin absorbs the carried start offset.  STRK_WD overrides (tuning only).
    int wd = local_search_range + step_size + 2;
    if (wd < 6) wd = 6;
    if (const char *env = getenv("STRK_WD")) {
        int v = atoi(env);
        if (v >= 1 && v <= 64) wd = v;
    }
    static const bool trace = getenv("STRK_RUN_TRACE") != nullptr;
    int ws = b->wide_short;
    if (const char *env = getenv("STRK_WIDE_SHORT")) ws = atoi(env) != 0;  // tuning only
    const int wd_cap = (STRK_MAX_WINDOW - 1) / 2 - 2;
    std::vector<int> h_read_ids, h_locus_ids;  // widening passes: the reads of the slots, the loci being redone
    std::vector<long long> h_slot_begin;
    std::vector<unsigned char> h_bin;
    float ms_dp = 0.f, ms_replay = 0.f;
    double acc[2] = {0, 0};  // [0] reference-equivalent cells, [1] executed cells

    // Where a widening pass has to look: per locus the carried-offset fractions its misses happened at (strk_slot_window)
    if (b->hint.reserve(2 * (size_t)(b->n_loci ? b->n_loci : 1)) != cudaSuccess) {
        cudaGetLastError();
        return set_err(STRK_ERR_NOMEM, "cannot allocate the window hints");
    }
    CU(cudaMemsetAsync(b->hint.p, 0, 2 * (size_t)b->n_loci * sizeof(double), st));

    for (int pass = 0;; ++pass) {
        if (wd > wd_cap) wd = wd_cap;
        const int threads = 256;
        // pass 0: every read of every locus; a widening pass: the reads of the loci being redone (next_loci)
        const long long n_slots = pass ? (long long)h_read_ids.size() : b->n_reads;
        const long long n_list = pass ? (long long)h_locus_ids.size() : b->n_loci;
        const int *d_read_ids = pass ? ctx->list_a.p : nullptr, *d_locus_ids = pass ? ctx->list_b.p : nullptr;
        const long long *d_slot_begin = pass ? ctx->list_c.p : nullptr;
        const double *d_hint = pass ? b->hint.p : nullptr;
        int W = 2 * strk_read_wd(wd, 1, ws) + 1;  // table stride: the widest per-read window
        if (pass) {
            // windows of a widening pass are stretched towards the starts the locus' offset has produced: measure the widest
            CU(cudaMemsetAsync(ctx->counter(Q_WIDEST), 0, sizeof(unsigned int), st));
            plan_reads_kernel<<<(unsigned)((n_slots + threads - 1) / threads), threads, 0, st>>>(
                d_read_ids, n_slots, b->d_seq_off, b->d_lens, b->d_est, b->d_read_locus, b->d_motif_off, b->d_motif_len, wd, ws,
                W, ctx->fams.p, ctx->d_acc + 1, nullptr, d_hint, ctx->counter(Q_WIDEST));
            CU(cudaGetLastError());
            unsigned int w_needed = 0;
            CU(cudaMemcpyAsync(&w_needed, ctx->counter(Q_WIDEST), sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            if ((int)w_needed > W) W = (int)w_needed;
            if (W > STRK_MAX_WINDOW)
                return set_err(STRK_ERR_SEARCH, "search left the widest supported window (%d sizes)", STRK_MAX_WINDOW);
        }
        if (ctx->fams.reserve((size_t)n_slots) != cudaSuccess || ctx->table.reserve((size_t)n_slots * (size_t)W) != cudaSuccess) {
            cudaGetLastError();
            return set_err(STRK_ERR_NOMEM, "cannot allocate score tables for %lld reads x %d sizes", n_slots, W);
        }
        const int b_len = b->ext.b_len();
        const int rowlen = b->ext.rowlen(pass ? W : strk_read_wd(wd, 1, ws));  // (n_hi - est <= W in a stretched window)
        plan_reads_kernel<<<(unsigned)((n_slots + threads - 1) / threads), threads, 0, st>>>(
            d_read_ids, n_slots, b->d_seq_off, b->d_lens, b->d_est, b->d_read_locus, b->d_motif_off, b->d_motif_len, wd,
            ws, W, ctx->fams.p, ctx->d_acc + 1, pass == 0 ? b->d_rep : nullptr, d_hint);
        CU(cudaGetLastError());
        ctx->stats[2] += 1;
        CU(cudaEventRecord(ctx->ev[0], st));
        int rc = STRK_OK;
        // packed kernel per rows-per-lane class, for every pass whose window it can hold (the first widening pass
        // included: 8x the first window); what it cannot take goes to the general kernel
        const bool use_packed = pk_window_ok(ctx, kernel, 0, W);
        DpPass dp{ctx->fams.p, b->d_arena, ctx->table.p, 0, b_len, rowlen, n_slots};
        if (!use_packed) {
            // (first pass: the work order lists the representatives only when identical reads share tables)
            dp.list[0] = pass ? nullptr : b->d_order;
            dp.cnt[0] = n_slots - (pass == 0 ? b->n_dup : 0);
        } else if (pass == 0) {  // the batch's work plan: the general kernel's reads, then one segment per class
            for (int k = 0; k < STRK_PK_NBIN; ++k) {
                dp.list[k] = b->d_order + b->bin_off[k], dp.cnt[k] = b->bin_cnt[k];
                dp.flank[k] = b->bin_flank[k], dp.mmax[k] = b->bin_mmax[k], dp.w[k] = W;
            }
            dp.list[0] = b->d_order, dp.cnt[0] = b->n_general;
        } else {
            rc = widening_pass(ctx, b, h_read_ids, h_bin, W, st, dp);
            if (rc) return rc;
        }
        long long n_packed = 0;
        rc = launch_pass(ctx, dp, st, &n_packed);
        if (rc) return rc;
        CU(cudaEventRecord(ctx->ev[1], st));
        CU(cudaMemsetAsync(ctx->counter(Q_MISS), 0, sizeof(unsigned int), st));
        CU(cudaMemsetAsync(ctx->counter(Q_MARGIN), 0, sizeof(unsigned int), st));
        rc = launch_replay(ctx, b, W, wd, ws, d_locus_ids, d_slot_begin, n_list, max_iters, local_search_range, step_size,
                           pass == 0 ? b->d_rep : nullptr, b->hint.p, st);
        if (rc) return rc;
        ctx->stats[2] += 1;
        CU(cudaEventRecord(ctx->ev[2], st));
        // [0] loci whose search left the window, [1] packed-kernel fallbacks, [2] loci saved by the wide_short margin
        unsigned int miss_fb[3] = {0, 0, 0};
        CU(cudaMemcpyAsync(miss_fb, ctx->counter(Q_MISS), 3 * sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(acc, ctx->d_acc, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));  // cumulative over passes
        CU(cudaStreamSynchronize(st));
        // (launch_pass zeroes the fallback counter of a pass with packed items only)
        const unsigned int miss = miss_fb[0], fallbacks = n_packed ? miss_fb[1] : 0;
        ctx->stats[6] += (double)(n_packed - (long long)fallbacks);
        ctx->stats[7] -= (double)(n_packed - (long long)fallbacks);
        float t0 = 0.f, t1 = 0.f;
        CU(cudaEventElapsedTime(&t0, ctx->ev[0], ctx->ev[1]));
        CU(cudaEventElapsedTime(&t1, ctx->ev[1], ctx->ev[2]));
        ms_dp += t0;
        ms_replay += t1;
        ctx->stats[7] += (double)(n_slots - (pass == 0 ? b->n_dup : 0));  // duplicates run no DP of their own
        if (trace)
            fprintf(stderr, "[strk_batch_run %p] pass %d: wd %d (wide_short %d, %d sizes), %lld reads of %lld loci, %s kernel, "
                    "dp %.3f ms, replay %.3f ms, %u loci left the window, %u used the margin, %u fallbacks\n", (void *)ctx, pass, wd, ws, W,
                    n_slots, n_list, use_packed ? "packed" : "general", t0, t1, miss, miss_fb[2], fallbacks);
        if (pass == 0 && b->n_loci >= 256) {  // policy for the next block filled into this batch object
            if (!ws && (long long)miss * 40 > b->n_loci) b->wide_short = 1;
            if (ws && (long long)(miss + miss_fb[2]) * 100 < b->n_loci) b->wide_short = 0;
        }
        if (miss == 0) break;

        // widening pass: redo the loci whose search left the window
        ctx->stats[5] += 1;
        if (wd >= wd_cap)
            return set_err(STRK_ERR_SEARCH, "search left the widest supported window (%d sizes)", STRK_MAX_WINDOW);
        rc = next_loci(ctx, b, pass == 0, max_iters, h_locus_ids, h_read_ids, h_slot_begin, st);
        if (rc) return rc;
        // The next pass looks where the misses happened (hints) with twice the margin; once that has not been enough twice
        // it widens 8x per pass like the blind scheme did (a search that goes nowhere near its start or its estimate).
        int widen = pass < 2 ? 2 : 8;
        if (const char *env = getenv("STRK_WIDEN1")) widen = pass == 0 && atoi(env) >= 2 ? atoi(env) : widen;  // tuning only
        wd *= widen;
    }
    ctx->stats[0] = acc[1];
    ctx->stats[1] = acc[0];
    ctx->stats[3] = ms_dp;
    ctx->stats[4] = ms_replay;
    return STRK_OK;
}

extern "C" int strk_batch_download(strk_ctx *ctx, strk_batch *b, int32_t *out) {
    if (!ctx || !b || (!out && b->n_reads)) return set_err(STRK_ERR_ARG, "strk_batch_download: null argument");
    CU(cudaSetDevice(ctx->device));
    if (b->n_reads) CU(cudaMemcpy(out, b->d_out, (size_t)b->n_reads * 4 * sizeof(int), cudaMemcpyDeviceToHost));
    return STRK_OK;
}

extern "C" int strk_count_reads_fmt(strk_ctx *ctx, int arena_format, const uint8_t *arena, uint64_t arena_bytes,
                                    const uint64_t *seq_off, const int32_t *lens, const int32_t *est_cn, int64_t n_reads,
                                    const int64_t *read_begin, const uint64_t *motif_off, const int32_t *motif_len,
                                    int64_t n_loci, int max_iters, int local_search_range, int step_size, int kernel,
                                    int32_t *out) {
    if (!ctx) return set_err(STRK_ERR_ARG, "strk_count_reads: null context");
    if (!ctx->reuse) ctx->reuse = new (std::nothrow) strk_batch();
    if (!ctx->reuse) return set_err(STRK_ERR_NOMEM, "out of host memory");
    strk_batch *b = ctx->reuse;  // device buffers are recycled across calls (no cudaMalloc per block of loci)
    int rc = batch_fill(ctx, b, arena, arena_bytes, seq_off, lens, est_cn, n_reads, read_begin, motif_off, motif_len,
                        n_loci, arena_format);
    if (rc) return rc;
    rc = strk_batch_run(ctx, b, max_iters, local_search_range, step_size, kernel, nullptr);
    if (!rc) rc = strk_batch_download(ctx, b, out);
    return rc;
}

extern "C" int strk_count_reads(strk_ctx *ctx, const uint8_t *arena, uint64_t arena_bytes, const uint64_t *seq_off,
                                const int32_t *lens, const int32_t *est_cn, int64_t n_reads, const int64_t *read_begin,
                                const uint64_t *motif_off, const int32_t *motif_len, int64_t n_loci, int max_iters,
                                int local_search_range, int step_size, int kernel, int32_t *out) {
    return strk_count_reads_fmt(ctx, STRK_ARENA_ASCII, arena, arena_bytes, seq_off, lens, est_cn, n_reads, read_begin,
                                motif_off, motif_len, n_loci, max_iters, local_search_range, step_size, kernel, out);
}

// The PyO3 function this library replaces, argument for argument (repeats.py:58-68): one read, strings in, four
// ints out.  A one-read batch through the same machinery (host-side planning, no device planning kernels).
extern "C" int strk_get_repeat_count(strk_ctx *ctx, int start_count, const char *tr_seq, int n_tr,
                                     const char *flank_left_seq, int n_fl, const char *flank_right_seq, int n_fr,
                                     const char *motif, int m, int max_iters, int local_search_range, int step_size,
                                     int use_shortcuts, int32_t out4[4]) {
    if (!ctx || !out4 || (n_tr && !tr_seq) || (n_fl && !flank_left_seq) || (n_fr && !flank_right_seq) || !motif)
        return set_err(STRK_ERR_ARG, "strk_get_repeat_count: null argument");
    if (n_tr < 0 || n_fl < 0 || n_fr < 0 || m <= 0) return set_err(STRK_ERR_ARG, "strk_get_repeat_count: bad length");
    if (use_shortcuts)
        return set_err(STRK_ERR_UNSUPPORTED, "use_shortcuts=True: the reference never passes it (repeats.py:67) and its "
                                             "semantics are not in the reference tree");
    std::vector<unsigned char> arena((size_t)n_fl + n_tr + n_fr + m);
    if (n_fl) memcpy(arena.data(), flank_left_seq, (size_t)n_fl);
    if (n_tr) memcpy(arena.data() + n_fl, tr_seq, (size_t)n_tr);
    if (n_fr) memcpy(arena.data() + n_fl + n_tr, flank_right_seq, (size_t)n_fr);
    memcpy(arena.data() + n_fl + n_tr + n_fr, motif, (size_t)m);
    const uint64_t seq_off = 0, motif_off = (uint64_t)n_fl + n_tr + n_fr;
    const int32_t lens[3] = {n_fl, n_tr, n_fr}, est = start_count, mlen = m;
    const int64_t read_begin[2] = {0, 1};
    int32_t row[4] = {0, 0, 0, 0};
    int rc = strk_count_reads_fmt(ctx, STRK_ARENA_ASCII, arena.data(), arena.size(), &seq_off, lens, &est, 1, read_begin,
                                  &motif_off, &mlen, 1, max_iters, local_search_range, step_size, STRK_KERNEL_AUTO, row);
    if (rc) return rc;
    out4[0] = row[0], out4[1] = row[1], out4[2] = row[2], out4[3] = row[0] - start_count;  // repeats.py:55-56
    return STRK_OK;
}

// ------------------------------------------------------------------------------------------------
// raw tables (parity checks of the DP itself) and the reference-boundary path
// ------------------------------------------------------------------------------------------------
// Device buffers of one call (the entry points below and alleles_api.cuh / realign_api.cuh).  Uploads are queued on
// `st`, the stream the call's kernels run on; on every way out, the destructor waits for `st` before it frees the
// buffers, so neither they nor the caller's host arrays are released under a queued copy or kernel.
struct TmpDev {
    cudaStream_t st;
    std::vector<void *> ptrs;
    ~TmpDev() {
        if (!ptrs.empty()) cudaStreamSynchronize(st);
        for (void *p : ptrs) cudaFree(p);
    }
    template <typename T>
    cudaError_t get(T **dst, size_t n) {
        cudaError_t e = cudaMalloc((void **)dst, (n ? n : 1) * sizeof(T));
        if (e == cudaSuccess) ptrs.push_back(*dst);
        return e;
    }
    template <typename T>
    cudaError_t up(T **dst, const T *src, size_t n) {
        cudaError_t e = get(dst, n);
        if (e == cudaSuccess && n) e = cudaMemcpyAsync(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice, st);
        return e;
    }
};

static int tables_common(strk_ctx *ctx, bool ref, const uint8_t *arena, uint64_t arena_bytes, const uint64_t *seq_off,
                         const int32_t *lens, const int32_t *motif_idx, const int32_t *n_lo, const int32_t *n_hi,
                         int64_t n_reads, const uint64_t *motif_off, const int32_t *motif_len, int64_t n_motifs,
                         const uint64_t *out_off, int kernel, void *out_host) {
    const char *who = ref ? "strk_ref_boundary_tables" : "strk_score_tables";
    if (!ctx || !arena || !seq_off || !lens || !n_lo || !n_hi || !motif_off || !motif_len || !out_off || !out_host)
        return set_err(STRK_ERR_ARG, "%s: null argument", who);
    if (n_reads <= 0 || n_reads > 0x7ffffff0LL) return set_err(STRK_ERR_ARG, "%s: bad family count", who);
    int rc = validate_reads(who, arena_bytes, seq_off, lens, n_reads);
    if (rc) return rc;
    rc = validate_motifs(who, arena_bytes, motif_off, motif_len, n_motifs);
    if (rc) return rc;
    CU(cudaSetDevice(ctx->device));
    std::vector<FamDesc> fams((size_t)n_reads);
    uint64_t total = 0;
    GenExtent ext = {};
    for (int64_t r = 0; r < n_reads; ++r) {
        const int64_t mi = motif_idx ? motif_idx[r] : r;
        if (mi < 0 || mi >= n_motifs) return set_err(STRK_ERR_ARG, "%s: motif index out of range", who);
        if (n_lo[r] < 0 || n_hi[r] < n_lo[r] || n_hi[r] > (1 << 22))
            return set_err(STRK_ERR_ARG, "%s: bad size window [%d, %d] for family %lld", who, n_lo[r], n_hi[r], (long long)r);
        FamDesc &f = fams[(size_t)r];
        f.db_off = seq_off[r];
        f.motif_off = motif_off[mi];
        f.out_off = out_off[r];
        f.n_fl = lens[3 * r];
        f.n_tr = lens[3 * r + 1];
        f.n_fr = lens[3 * r + 2];
        f.m = motif_len[mi];
        f.n_lo = n_lo[r];
        f.n_hi = n_hi[r];
        // an empty candidate has no alignment (parasail rejects empty sequences)
        if (ref && f.n_lo == 0 && (f.n_fl == 0 || f.n_fr == 0))
            return set_err(STRK_ERR_ARG, "%s: family %lld scores an empty candidate (n = 0 with an empty flank)", who,
                           (long long)r);
        if (!ref && f.n_lo == 0 && f.n_fl + f.n_fr == 0)
            return set_err(STRK_ERR_ARG, "%s: family %lld scores an empty candidate (n = 0 without flanks)", who,
                           (long long)r);
        const int64_t cols = (int64_t)std::max(f.n_fl, f.n_fr) + (int64_t)f.m * f.n_hi;
        if (cols > (1 << 26)) return set_err(STRK_ERR_ARG, "%s: candidate too long", who);
        ext.add(f.n_fl, f.n_fr, f.n_fl + f.n_tr + f.n_fr, f.m, f.n_hi);  // (rowlen(0): a table has no window margin)
        total = std::max<uint64_t>(total, out_off[r] + (uint64_t)(f.n_hi - f.n_lo + 1));
    }
    const int b_len = ext.b_len(), rowlen = ext.rowlen(0);
    // same routing as the batch paths: packed kernel per class, the rest (and its fallbacks) to the general kernel
    ClassLists lists;
    for (int64_t r = 0; r < n_reads; ++r) {
        const FamDesc &f = fams[(size_t)r];
        const int w = f.n_hi - f.n_lo + 1;
        lists.add(pk_class(ctx, kernel, ref, w, f.n_fl, f.n_tr, f.n_fr, f.m), (int)r, f.m, f.n_fl, f.n_fr, w);
    }
    TmpDev tmp{ctx->stream};
    unsigned char *d_arena = nullptr, *d_table = nullptr;
    FamDesc *d_fams = nullptr;
    cudaError_t e = tmp.up(&d_arena, arena, (size_t)arena_bytes);
    if (e == cudaSuccess) e = tmp.up(&d_fams, fams.data(), fams.size());
    if (e == cudaSuccess) e = tmp.get(&d_table, (size_t)total * (ref ? 2 * sizeof(long long) : sizeof(int)));
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(STRK_ERR_NOMEM, "%s: %s", who, cudaGetErrorString(e));
    }
    for (int k = 0; k < 8; ++k) ctx->stats[k] = 0;
    DpPass p{d_fams, d_arena, d_table, ref ? 1 : 0, b_len, rowlen, n_reads};
    if (lists.items[0].size() == (size_t)n_reads) {
        p.cnt[0] = n_reads;  // every family on the general kernel, in order
    } else {
        rc = lists.upload(ctx->list_d, ctx->stream, p);
        if (rc) return rc;
    }
    long long n_packed = 0;
    rc = launch_pass(ctx, p, ctx->stream, &n_packed);
    if (rc) return rc;
    if (n_packed) {
        unsigned int fb = 0;
        CU(cudaMemcpyAsync(&fb, ctx->counter(Q_FALLBACK), sizeof(unsigned int), cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        ctx->stats[6] = (double)(n_packed - (long long)fb);
    }
    ctx->stats[7] = (double)n_reads - ctx->stats[6];
    CU(cudaStreamSynchronize(ctx->stream));
    if (!ref) {
        CU(cudaMemcpy(out_host, d_table, (size_t)total * sizeof(int), cudaMemcpyDeviceToHost));
    } else {
        // unpack (score, end_query) pairs: the device layout per family is [fwd keys W][rev keys W]
        std::vector<long long> keys((size_t)total * 2);
        CU(cudaMemcpy(keys.data(), d_table, keys.size() * sizeof(long long), cudaMemcpyDeviceToHost));
        int32_t *o = (int32_t *)out_host;
        for (int64_t r = 0; r < n_reads; ++r) {
            const FamDesc &f = fams[(size_t)r];
            const int W = f.n_hi - f.n_lo + 1;
            const long long *k0 = keys.data() + 2 * f.out_off;
            for (int k = 0; k < W; ++k) {
                int fs, fe, rs, re;
                ref_unpack(k0[k], fs, fe);
                ref_unpack(k0[W + k], rs, re);
                int32_t *dst = o + 4 * (f.out_off + (uint64_t)k);
                dst[0] = fs, dst[1] = fe, dst[2] = rs, dst[3] = re;
            }
        }
    }
    return STRK_OK;
}

extern "C" int strk_score_tables(strk_ctx *ctx, const uint8_t *arena, uint64_t arena_bytes, const uint64_t *seq_off,
                                 const int32_t *lens, const int32_t *motif_idx, const int32_t *n_lo, const int32_t *n_hi,
                                 int64_t n_reads, const uint64_t *motif_off, const int32_t *motif_len, int64_t n_motifs,
                                 const uint64_t *out_off, int kernel, int32_t *scores) {
    return tables_common(ctx, false, arena, arena_bytes, seq_off, lens, motif_idx, n_lo, n_hi, n_reads, motif_off,
                         motif_len, n_motifs, out_off, kernel, scores);
}

extern "C" int strk_ref_boundary_tables(strk_ctx *ctx, const uint8_t *arena, uint64_t arena_bytes,
                                        const uint64_t *seq_off, const int32_t *lens, const int32_t *n_lo,
                                        const int32_t *n_hi, int64_t n_loci, const uint64_t *motif_off,
                                        const int32_t *motif_len, const uint64_t *out_off, int kernel, int32_t *out) {
    return tables_common(ctx, true, arena, arena_bytes, seq_off, lens, nullptr, n_lo, n_hi, n_loci, motif_off, motif_len,
                         n_loci, out_off, kernel, out);
}

// First window of the boundary search: start +- max(6, range + step + 2) sizes, like the read path's (a search that
// starts where it ends touches start +- (range + step)); one that leaves it is redone 4x wider.  Measured on 32 768
// HiFi-sized windows: +- 9 sizes 3.89 ms, +- 7 3.79 ms, +- 6 3.33 ms per block.  STRK_REF_WD=<n> raises the floor of 6
// (tuning only).
static int ref_first_wd(int range, int step) {
    static const int wd_env = getenv("STRK_REF_WD") ? atoi(getenv("STRK_REF_WD")) : 6;
    return std::max(wd_env > 0 ? wd_env : 6, range + step + 2);
}

// The first steps of strk_ref_counts: argument checks, the first boundary window of every locus (ctx->ref.h_wd), the
// context's reference buffers, and the upload of the inputs with phase 1's results cleared, queued on `st`.
static int ref_setup(strk_ctx *ctx, cudaStream_t st, const uint8_t *arena, uint64_t arena_bytes, const uint64_t *seq_off,
                     const int32_t *lens, const int32_t *start_count, const int32_t *ref_size, const int32_t *rc_params,
                     int64_t n_loci, const uint64_t *motif_off, const int32_t *motif_len) {
    int rc = validate_reads("strk_ref_counts", arena_bytes, seq_off, lens, n_loci);
    if (rc) return rc;
    rc = validate_motifs("strk_ref_counts", arena_bytes, motif_off, motif_len, n_loci);
    if (rc) return rc;
    RefBufs &d = ctx->ref;
    const size_t n = (size_t)n_loci;
    d.h_wd.resize(n);
    for (size_t l = 0; l < n; ++l) {
        if (strk_check_est(start_count[l], motif_len[l]) || rc_params[3 * l] < 0 || rc_params[3 * l + 1] < 0 ||
            rc_params[3 * l + 2] < 0 || rc_params[3 * l + 1] > 1000 || rc_params[3 * l + 2] > 1000)
            return set_err(STRK_ERR_ARG, "strk_ref_counts: bad start count / search parameters for locus %lld", (long long)l);
        d.h_wd[l] = ref_first_wd(rc_params[3 * l + 1], rc_params[3 * l + 2]);
    }
    CU(cudaSetDevice(ctx->device));
    for (int k = 0; k < 8; ++k) ctx->stats[k] = 0;
    cudaError_t e = d.arena.reserve((size_t)arena_bytes);
    if (e == cudaSuccess) e = d.seq_off.reserve(n);
    if (e == cudaSuccess) e = d.motif_off.reserve(n);
    for (DevBuf<int> *p : {&d.lens, &d.rc})
        if (e == cudaSuccess) e = p->reserve(3 * n);
    // (lists: every class-list upload of the call then fits, and none reallocates a buffer a queued pass still reads)
    for (DevBuf<int> *p : {&d.start, &d.ref_size, &d.motif_len, &d.wd, &d.l_off, &d.r_off, &d.n_off, &d.ids_a, &d.ids_b,
                           &d.tier_ids, &d.lists})
        if (e == cudaSuccess) e = p->reserve(n);
    if (e == cudaSuccess) e = d.cnt.reserve(8);
    if (e == cudaSuccess) e = d.out.reserve(8 * n + 8);
    if (e == cudaSuccess) e = d.redo.reserve(n);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(STRK_ERR_NOMEM, "strk_ref_counts: %s", cudaGetErrorString(e));
    }
    CU(cudaMemcpyAsync(d.arena.p, arena, (size_t)arena_bytes, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d.seq_off.p, seq_off, n * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d.motif_off.p, motif_off, n * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d.lens.p, lens, 3 * n * sizeof(int), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d.start.p, start_count, n * sizeof(int), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d.ref_size.p, ref_size, n * sizeof(int), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d.rc.p, rc_params, 3 * n * sizeof(int), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d.motif_len.p, motif_len, n * sizeof(int), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d.wd.p, d.h_wd.data(), n * sizeof(int), cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(d.l_off.p, 0, n * sizeof(int), st));
    CU(cudaMemsetAsync(d.r_off.p, 0, n * sizeof(int), st));
    CU(cudaMemsetAsync(d.n_off.p, 0, n * sizeof(int), st));
    return STRK_OK;
}

// One widening round of phase 1: the loci of `ids` (n of them; with d_n, the first min(n, *d_n)) at the windows
// ref_replay1_kernel raised for them (d.wd, at most wd sizes either side) through the general kernel, then replayed.
// Those that leave their window again are appended to `again`; `cnt` gets the counters of ref_replay1_kernel.
static int ref_widen(strk_ctx *ctx, const int *ids, int n, const unsigned int *d_n, int wd, int *again, unsigned int *cnt,
                     int b_len, int rowlen, int vcf_anchor_size) {
    RefBufs &d = ctx->ref;
    cudaStream_t st = ctx->stream;
    const int T = 128, WD_MAX = (STRK_MAX_WINDOW - 1) / 2;
    ref_plan1_kernel<<<(unsigned)((n + T - 1) / T), T, 0, st>>>(ids, n, d.seq_off.p, d.lens.p, d.start.p, d.wd.p, d.motif_off.p,
                                                               d.motif_len.p, 2 * wd + 1, ctx->fams.p, d_n);
    CU(cudaGetLastError());
    int rc = launch_general(ctx, true, ctx->fams.p, nullptr, n, d.arena.p, ctx->table64.p, b_len, rowlen, st, d_n);
    if (rc) return rc;
    ref_replay1_kernel<<<(unsigned)((n + T - 1) / T), T, 0, st>>>(ids, n, ctx->table64.p, ctx->fams.p, d.start.p, d.rc.p,
                                                                 d.ref_size.p, vcf_anchor_size, WD_MAX, d.wd.p, d.l_off.p,
                                                                 d.r_off.p, d.n_off.p, again, cnt, d_n);
    CU(cudaGetLastError());
    return STRK_OK;
}

// The errors of a phase 1 pass, from the counters of ref_replay1_kernel
static int ref_search_error(const unsigned int *cnt, const int32_t *rc_params) {
    if (cnt[2])
        return set_err(STRK_ERR_SEARCH, "strk_ref_counts: locus %lld left the widest window", (long long)(0x7fffffffu - cnt[2]));
    if (cnt[1]) {
        const long long l = (long long)(0x7fffffffu - cnt[1]);
        return set_err(STRK_ERR_SEARCH, "strk_ref_counts: locus %lld scored no size (max_iters = %d)", l, rc_params[3 * l]);
    }
    return STRK_OK;
}

// get_ref_repeat_count (repeats.py:73-192) for a batch of loci, device-resident from upload to results.
// Phase 1 (skipped with respect_coords, repeats.py:99): boundary tables (two sg_qe sweeps per locus, every candidate
// size of a window at once: the packed kernel in reference mode) + the dual-score search replayed one thread per locus
// -> l_offset / r_offset; a second look redoes up to CAP2 loci whose search left the first window 4x wider.  Phase 2:
// the final count on the adjusted flanks = the read-path kernels (packed kernel, device replay) with one "read" per
// locus, one pass per search-parameter tier, and a kernel that assembles the 8 result ints per locus.  Everything is
// queued on the context's stream; ONE synchronisation brings back the results and the flags of the loci the device did
// not settle (a search that left the window of the second look, or of phase 2).  The host finishes those, on the
// buffers already resident: phase 1 4x wider per round, then phase 2 through strk_batch_run, which widens as far as a
// search needs.  (Every host synchronisation of a call under another context's read kernels waits for SM slots that
// the persistent read CTAs free only at the end of a class launch.)
extern "C" int strk_ref_counts(strk_ctx *ctx, const uint8_t *arena, uint64_t arena_bytes, const uint64_t *seq_off,
                               const int32_t *lens, const int32_t *start_count, const int32_t *ref_size,
                               const int32_t *rc_params, int64_t n_loci, const uint64_t *motif_off,
                               const int32_t *motif_len, int vcf_anchor_size, int respect_coords, int32_t *out) {
    if (!ctx || !arena || !seq_off || !lens || !start_count || !ref_size || !rc_params || !motif_off || !motif_len || !out)
        return set_err(STRK_ERR_ARG, "strk_ref_counts: null argument");
    if (n_loci <= 0 || n_loci > 0x7ffffff0LL) return set_err(STRK_ERR_ARG, "strk_ref_counts: bad locus count");
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t_begin = now();
    cudaStream_t st = ctx->stream;
    int rc = ref_setup(ctx, st, arena, arena_bytes, seq_off, lens, start_count, ref_size, rc_params, n_loci, motif_off,
                       motif_len);
    if (rc) return rc;
    RefBufs &d = ctx->ref;
    const size_t n = (size_t)n_loci;
    const bool phase1 = !respect_coords;
    const int CAP2 = 4096, WD_MAX = (STRK_MAX_WINDOW - 1) / 2, T = 128;
    // phase 1's table stride: the widest first window; the second look's: 4x that
    const int wd1 = *std::max_element(d.h_wd.begin(), d.h_wd.end()), stride_w = 2 * wd1 + 1;
    const int wd1b = std::min(WD_MAX, 4 * wd1), stride_w2 = 2 * wd1b + 1;

    // ---- host plan: phase 1's classes, scratch maxima, the tiers in first-appearance order
    GenExtent ext = {};
    int wd2_max = 0;
    double cells1 = 0.0;
    ClassLists &lists = d.classes;
    lists.clear();
    size_t n_tiers = 0;
    for (int64_t l = 0; l < n_loci; ++l) {
        const int fl = lens[3 * l], tr = lens[3 * l + 1], fr = lens[3 * l + 2], m = motif_len[l];
        const int n1 = fl + tr + fr;
        // the longest candidate prefix of either phase (phase 2 moves at most both flanks into the tract:
        // (fl + fr) / m + 1 more copies)
        ext.add(fl, fr, n1, m, start_count[l] + (fl + fr) / m + 1);
        if (phase1) {  // executed cells of the first pass: two sweeps of db x (flank + motif * n_hi)
            lists.add(pk_class(ctx, STRK_KERNEL_AUTO, 1, stride_w, fl, tr, fr, m), (int)l, m, fl, fr, stride_w);
            cells1 += (double)n1 * ((double)fl + fr + 2.0 * m * ((double)start_count[l] + d.h_wd[(size_t)l]));
        }
        const int32_t *p = rc_params + 3 * l;
        size_t t = 0;
        while (t < n_tiers && !std::equal(p, p + 3, d.tiers[t].rc)) ++t;
        if (t == n_tiers) {
            if (n_tiers == d.tiers.size()) d.tiers.emplace_back();
            RefTier &nt = d.tiers[n_tiers++];
            std::copy(p, p + 3, nt.rc);
            nt.wd2 = std::max(6, p[1] + p[2] + 2);  // the read path's first window
            nt.W2 = 2 * nt.wd2 + 1;
            nt.ids.clear();
            nt.classes.clear();
            wd2_max = std::max(wd2_max, nt.wd2);
        }
        d.tiers[t].ids.push_back((int)l);
    }
    d.tiers.resize(n_tiers);  // (the vectors of the tiers kept keep their capacity for the next call)
    // one tier classed like phase 1: phase 2 takes phase 1's lists (moving bases between flank and tract does not change
    // a window's class), slot q = locus q
    const bool reuse = phase1 && d.tiers.size() == 1 &&
                       pk_window_ok(ctx, STRK_KERNEL_AUTO, 1, stride_w) == pk_window_ok(ctx, STRK_KERNEL_AUTO, 0, d.tiers[0].W2);
    size_t table2 = 0;
    for (RefTier &t : d.tiers) {
        table2 = std::max(table2, t.ids.size() * (size_t)t.W2);
        for (size_t q = 0; q < t.ids.size() && !reuse; ++q) {
            const int l = t.ids[q];
            const int fl = lens[3 * l], tr = lens[3 * l + 1], fr = lens[3 * l + 2], m = motif_len[l];
            t.classes.add(pk_class(ctx, STRK_KERNEL_AUTO, 0, t.W2, fl, tr, fr, m), (int)q, m, fl, fr, t.W2);
        }
    }
    const int b_len = ext.b_len(), rowlen = ext.rowlen(std::max(std::max(wd1, wd2_max), wd1b));

    // ---- device buffers (context-owned, recycled)
    if (!ctx->ref_batch) ctx->ref_batch = new (std::nothrow) strk_batch();
    if (!ctx->ref_batch) return set_err(STRK_ERR_NOMEM, "out of host memory");
    strk_batch *b = ctx->ref_batch;
    cudaError_t e = batch_bind(b, (long long)n, (long long)n);
    if (e == cudaSuccess) e = ctx->fams.reserve(std::max(n, (size_t)CAP2));
    if (e == cudaSuccess) e = ctx->table64.reserve(std::max(n * (size_t)stride_w * 2, (size_t)CAP2 * (size_t)stride_w2 * 2));
    if (e == cudaSuccess) e = ctx->table.reserve(table2);
    if (e == cudaSuccess) e = ctx->fallback.reserve(n);  // (for every pass of the call: see launch_pass)
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(STRK_ERR_NOMEM, "strk_ref_counts: %s", cudaGetErrorString(e));
    }
    b->d_arena = d.arena.p;
    DpPass p1{ctx->fams.p, d.arena.p, ctx->table64.p, 1, b_len, rowlen, n_loci};
    if (phase1) {
        rc = lists.upload(d.lists, st, p1);
        if (rc) return rc;
    }
    CU(cudaMemsetAsync(d.cnt.p, 0, 8 * sizeof(unsigned int), st));
    CU(cudaMemsetAsync(ctx->d_acc, 0, 4 * sizeof(double), st));

    // ---- phase 1, then the second look: the loci whose search left the first window (a percent of a block at +-6
    // sizes), listed and counted on the device (ids_a, cnt[0]), up to CAP2 of them 4x wider; the rest keep their flag
    if (phase1) {
        ref_plan1_kernel<<<(unsigned)((n + T - 1) / T), T, 0, st>>>(nullptr, (int)n, d.seq_off.p, d.lens.p, d.start.p, d.wd.p,
                                                                   d.motif_off.p, d.motif_len.p, stride_w, ctx->fams.p);
        CU(cudaGetLastError());
        CU(cudaEventRecord(ctx->ev[0], st));
        long long n_packed = 0;
        rc = launch_pass(ctx, p1, st, &n_packed);
        if (rc) return rc;
        CU(cudaEventRecord(ctx->ev[1], st));
        ref_replay1_kernel<<<(unsigned)((n + T - 1) / T), T, 0, st>>>(nullptr, (int)n, ctx->table64.p, ctx->fams.p, d.start.p,
                                                                     d.rc.p, d.ref_size.p, vcf_anchor_size, WD_MAX, d.wd.p,
                                                                     d.l_off.p, d.r_off.p, d.n_off.p, d.ids_a.p, d.cnt.p);
        CU(cudaGetLastError());
        ref_clamp_count_kernel<<<1, 32, 0, st>>>(d.cnt.p, (unsigned)CAP2);
        rc = ref_widen(ctx, d.ids_a.p, CAP2, d.cnt.p, wd1b, d.ids_b.p, d.cnt.p + 4, b_len, rowlen, vcf_anchor_size);
        if (rc) return rc;
    }

    // ---- phase 2, one pass per tier in stream order (each overwrites ctx->table and the slots of the batch); loci whose
    // phase 1 is not final yet run with their unadjusted flanks and are flagged
    size_t at = 0;
    for (size_t t = 0; t < d.tiers.size(); ++t) {
        RefTier &tier = d.tiers[t];
        const int nt = (int)tier.ids.size();
        DpPass p2{ctx->fams.p, d.arena.p, ctx->table.p, 0, b_len, rowlen, nt};
        int *ids = nullptr;
        if (reuse) {  // phase 1's classes at phase 2's window
            p2 = p1, p2.table = ctx->table.p, p2.ref_mode = 0;
            std::fill_n(p2.w, STRK_PK_NBIN, tier.W2);
        } else {
            ids = d.tier_ids.p + at;
            CU(cudaMemcpyAsync(ids, tier.ids.data(), nt * sizeof(int), cudaMemcpyHostToDevice, st));
            rc = tier.classes.upload(d.lists, st, p2);
            if (rc) return rc;
        }
        at += (size_t)nt;
        ref_plan2_kernel<<<(unsigned)((nt + T - 1) / T), T, 0, st>>>(ids, nt, d.seq_off.p, d.lens.p, d.start.p, d.motif_off.p,
                                                                    d.motif_len.p, d.l_off.p, d.r_off.p, b->d_seq_off,
                                                                    b->d_lens, b->d_est, b->d_motif_off, b->d_motif_len,
                                                                    b->d_read_begin, b->d_read_locus);
        CU(cudaGetLastError());
        plan_reads_kernel<<<(unsigned)((nt + 255) / 256), 256, 0, st>>>(nullptr, (long long)nt, b->d_seq_off, b->d_lens,
                                                                       b->d_est, b->d_read_locus, b->d_motif_off,
                                                                       b->d_motif_len, tier.wd2, 0, tier.W2, ctx->fams.p,
                                                                       ctx->d_acc + 1, nullptr);
        CU(cudaGetLastError());
        if (t == 0) CU(cudaEventRecord(ctx->ev[2], st));
        long long n_packed = 0;
        rc = launch_pass(ctx, p2, st, &n_packed);
        if (rc) return rc;
        if (t + 1 == d.tiers.size()) CU(cudaEventRecord(ctx->ev[3], st));
        rc = launch_replay(ctx, b, tier.W2, tier.wd2, 0, nullptr, nullptr, nt, tier.rc[0], tier.rc[1], tier.rc[2], nullptr,
                           nullptr, st);
        if (rc) return rc;
        ref_assemble_kernel<<<(unsigned)((nt + T - 1) / T), T, 0, st>>>(ids, nt, b->d_out, b->d_status, d.lens.p, d.l_off.p,
                                                                       d.r_off.p, d.n_off.p, d.out.p, d.redo.p);
        CU(cudaGetLastError());
    }
    CU(cudaEventRecord(ctx->ev[4], st));

    // ---- the one synchronisation: results, flags, counters
    std::vector<unsigned char> flags(n);
    unsigned int h_cnt[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    double acc[2] = {0, 0};
    CU(cudaMemcpyAsync(out, d.out.p, 8 * n * sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(flags.data(), d.redo.p, n, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h_cnt, d.cnt.p, sizeof(h_cnt), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(acc, ctx->d_acc, sizeof(acc), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    rc = ref_search_error(h_cnt, rc_params);
    if (!rc) rc = ref_search_error(h_cnt + 4, rc_params);
    if (rc) return rc;
    // DP kernels: ev 0-1 (phase 1), 2-3 (phase 2; with several tiers, the replays between them too); replay, second look
    // and planning kernels: ev 1-2, 3-4
    float ms[4] = {0.f, 0.f, 0.f, 0.f};
    for (int k = phase1 ? 0 : 2; k < 4; ++k) CU(cudaEventElapsedTime(&ms[k], ctx->ev[k], ctx->ev[k + 1]));
    ctx->stats[0] = cells1 + acc[1];
    ctx->stats[1] = acc[0];
    ctx->stats[2] += (phase1 ? 3 : 0) + 4 * (double)d.tiers.size();  // (launch_* count their own)
    ctx->stats[3] = ms[0] + ms[2];
    ctx->stats[4] = ms[1] + ms[3];

    // ---- host finish of the flagged loci
    std::vector<int> redo, ids;
    for (size_t l = 0; l < n; ++l)
        if (flags[l]) redo.push_back((int)l);
    const double t_finish = now();
    if (!redo.empty()) {
        // phase 1 not final (n_off < 0): 4x wider per round; no window is wider than 16x the first one yet
        for (int l : redo)
            if (out[8 * (size_t)l + 4] < 0) ids.push_back(l);
        int *d_ids = d.ids_a.p, *d_again = d.ids_b.p;
        unsigned int n_pending = (unsigned int)ids.size();
        if (n_pending) CU(cudaMemcpyAsync(d_ids, ids.data(), ids.size() * sizeof(int), cudaMemcpyHostToDevice, st));
        for (int wd = std::min(WD_MAX, 16 * wd1); n_pending > 0; wd = std::min(WD_MAX, 4 * wd)) {
            if (ctx->fams.reserve(n_pending) != cudaSuccess ||
                ctx->table64.reserve((size_t)n_pending * (size_t)(2 * wd + 1) * 2) != cudaSuccess) {
                cudaGetLastError();
                return set_err(STRK_ERR_NOMEM, "strk_ref_counts: cannot allocate the boundary tables");
            }
            CU(cudaMemsetAsync(d.cnt.p, 0, 4 * sizeof(unsigned int), st));
            CU(cudaEventRecord(ctx->ev[0], st));
            rc = ref_widen(ctx, d_ids, (int)n_pending, nullptr, wd, d_again, d.cnt.p, b_len, ext.rowlen(wd), vcf_anchor_size);
            if (rc) return rc;
            CU(cudaEventRecord(ctx->ev[1], st));
            unsigned int c[4] = {0, 0, 0, 0};
            CU(cudaMemcpyAsync(c, d.cnt.p, sizeof(c), cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            rc = ref_search_error(c, rc_params);
            if (rc) return rc;
            float t_round = 0.f;
            CU(cudaEventElapsedTime(&t_round, ctx->ev[0], ctx->ev[1]));
            ctx->stats[2] += 2;
            ctx->stats[4] += t_round;
            n_pending = c[0];
            std::swap(d_ids, d_again);
        }
        // phase 2 of every flagged locus, per tier (strk_batch_run counts its own run only)
        double keep[8];
        memcpy(keep, ctx->stats, sizeof(keep));
        for (const RefTier &tier : d.tiers) {
            ids.clear();
            for (int l : tier.ids)
                if (flags[(size_t)l]) ids.push_back(l);
            if (ids.empty()) continue;
            const int nt = (int)ids.size();
            e = batch_bind(b, nt, nt);
            if (e != cudaSuccess) {
                cudaGetLastError();
                return set_err(STRK_ERR_NOMEM, "strk_ref_counts: %s", cudaGetErrorString(e));
            }
            b->d_arena = d.arena.p;
            b->h_read_begin.resize((size_t)nt + 1);
            for (int q = 0; q <= nt; ++q) b->h_read_begin[(size_t)q] = q;
            CU(cudaMemcpyAsync(d.ids_a.p, ids.data(), nt * sizeof(int), cudaMemcpyHostToDevice, st));
            ref_plan2_kernel<<<(unsigned)((nt + T - 1) / T), T, 0, st>>>(d.ids_a.p, nt, d.seq_off.p, d.lens.p, d.start.p,
                                                                        d.motif_off.p, d.motif_len.p, d.l_off.p, d.r_off.p,
                                                                        b->d_seq_off, b->d_lens, b->d_est, b->d_motif_off,
                                                                        b->d_motif_len, b->d_read_begin);
            CU(cudaGetLastError());
            CU(cudaStreamSynchronize(st));  // batch_plan reads the batch on the fill stream
            rc = batch_plan(ctx, b, arena_bytes);
            if (rc) return rc;
            rc = strk_batch_run(ctx, b, tier.rc[0], tier.rc[1], tier.rc[2], STRK_KERNEL_AUTO, nullptr);
            if (rc) return rc;
            for (int k = 0; k < 8; ++k) keep[k] += ctx->stats[k];
            ref_assemble_kernel<<<(unsigned)((nt + T - 1) / T), T, 0, st>>>(d.ids_a.p, nt, b->d_out, b->d_status, d.lens.p,
                                                                           d.l_off.p, d.r_off.p, d.n_off.p, d.out.p, d.redo.p);
            CU(cudaGetLastError());
            keep[2] += 2;
        }
        CU(cudaMemcpyAsync(out, d.out.p, 8 * n * sizeof(int), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        memcpy(ctx->stats, keep, sizeof(keep));
    }
    ctx->stats[5] = (double)redo.size();  // loci finished on the host
    if (getenv("STRK_REF_TIMING"))
        fprintf(stderr, "[strk_ref_counts] %lld loci, %zu tiers: DP kernels %.2f + %.2f ms, replay / second look / planning "
                "kernels %.2f + %.2f ms (device clock), %u loci took the second look; %zu finished on the host in %.2f ms, "
                "%.2f ms in all (host clock)\n", (long long)n_loci, d.tiers.size(), ms[0], ms[2], ms[1], ms[3], h_cnt[0],
                redo.size(), now() - t_finish, now() - t_begin);
    return STRK_OK;
}

// ------------------------------------------------------------------------------------------------
// integer issue-rate micro-benchmark (roofline denominator)
// ------------------------------------------------------------------------------------------------
extern "C" int strk_measure_int_peak(strk_ctx *ctx, double out_tiops[3]) {
    if (!ctx || !out_tiops) return set_err(STRK_ERR_ARG, "strk_measure_int_peak: null argument");
    CU(cudaSetDevice(ctx->device));
    int *d_out = (int *)ctx->counter(Q_INT_PEAK);  // context-owned scratch word and events: nothing to release on an error path
    const int grid = ctx->n_sm * 8, threads = 256, iters = 4096;
    const double instr = (double)grid * threads * (double)iters * 64.0;  // lane-level integer instructions
    cudaEvent_t e0 = ctx->ev[0], e1 = ctx->ev[1];
    for (int mode = 0; mode < 3; ++mode) {
        float best = 1e30f;
        for (int rep = 0; rep < 4; ++rep) {
            CU(cudaEventRecord(e0, ctx->stream));
            if (mode == 0) int_peak_kernel<0><<<grid, threads, 0, ctx->stream>>>(iters, rep + 3, d_out);
            if (mode == 1) int_peak_kernel<1><<<grid, threads, 0, ctx->stream>>>(iters, rep + 3, d_out);
            if (mode == 2) int_peak_kernel<2><<<grid, threads, 0, ctx->stream>>>(iters, rep + 3, d_out);
            CU(cudaGetLastError());
            CU(cudaEventRecord(e1, ctx->stream));
            CU(cudaEventSynchronize(e1));
            float ms = 0.f;
            CU(cudaEventElapsedTime(&ms, e0, e1));
            if (rep > 0 && ms < best) best = ms;
        }
        out_tiops[mode] = instr / ((double)best * 1e-3) / 1e12;
    }
    return STRK_OK;
}

// ------------------------------------------------------------------------------------------------
// bootstrap / GMM allele calls (the consumer of the per-read counts; SURVEY 8f N3)
// ------------------------------------------------------------------------------------------------
#include "alleles_api.cuh"
#include "realign_api.cuh"

#if PK_PHASE_TIMERS
// Measurement build only (not in include/strkit_b200.h): copies the packed kernel's phase timers of `device` to
// out[2 * 2 * 17 * 4] (the layout of pk_phase_clk in dp_packed.cuh) and, with reset != 0, clears them.
extern "C" int strk_pk_phase_timers(int device, unsigned long long *out, int reset) {
    if (!out) return set_err(STRK_ERR_ARG, "strk_pk_phase_timers: null argument");
    CU(cudaSetDevice(device));
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpyFromSymbol(out, pk_phase_clk, sizeof(pk_phase_clk)));
    if (reset) {
        static const unsigned long long zero[2 * 2 * 17 * 4] = {0ull};
        CU(cudaMemcpyToSymbol(pk_phase_clk, zero, sizeof(pk_phase_clk)));
    }
    return STRK_OK;
}
#endif
