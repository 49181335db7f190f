// alleles_api.cuh -- C entry points of the bootstrap / GMM allele caller (included at the end of api.cu, which
// defines strk_ctx, set_err and CU).  Declarations and the reference lines they replace: include/strkit_b200.h.
#pragma once
#include <type_traits>

#include "alleles.cuh"

// per_locus: the allele counts come per locus (validated by the caller) and n_alleles is 0; else n_alleles is the
// batch-wide count, 1 or 2
static int alleles_params(AlleleParams *P, int n_alleles, bool per_locus, int num_bootstrap, int min_reads,
                          int min_allele_reads, int force_gm_filter, double expansion_ratio, int filter_factor,
                          int n_init, uint64_t seed) {
    if (per_locus ? n_alleles != 0 : (n_alleles < 1 || n_alleles > 2))
        return set_err(STRK_ERR_UNSUPPORTED, "call_alleles: n_alleles = %d (1 and 2 are implemented)", n_alleles);
    if (num_bootstrap < 2 || num_bootstrap > ALL_MAX_BOOT)  // the reference itself fails for 1 (allele.py:163-167,258)
        return set_err(STRK_ERR_ARG, "call_alleles: num_bootstrap must be in 2..%d", ALL_MAX_BOOT);
    if (n_init < 1 || n_init > ALL_N_INIT_MAX || filter_factor < 1)
        return set_err(STRK_ERR_ARG, "call_alleles: bad GMM parameters (n_init %d, filter_factor %d)", n_init, filter_factor);
    P->n_alleles = n_alleles;
    P->num_bootstrap = num_bootstrap;
    P->min_reads = min_reads;
    P->n_init = n_init;
    P->max_iter = 100;
    P->force_gm_filter = force_gm_filter;
    P->tol = 1e-3;
    P->reg_covar = 1e-6;
    P->allele_filter = ((double)min_allele_reads - 0.1) / (double)num_bootstrap;
    P->expansion_ratio = expansion_ratio;
    P->filter_weight = 1.0 / ((double)filter_factor * 2.0);
    P->filter_factor = filter_factor;
    P->small_allele_min = 8.0;
    P->seed = seed;
    return STRK_OK;
}

// a kernel's dynamic shared memory plus its static arrays must fit the launch: above 48 KB in all the kernel opts in
// to the larger carve-out (the aggregation's sort keys take 48 KB at 4096 replicates; the deep kernels' tables)
template <class Kernel>
static cudaError_t smem_opt_in(Kernel kernel, size_t dyn) {
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, kernel);
    if (e == cudaSuccess && dyn + fa.sharedSizeBytes > 48 * 1024)
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
    return e;
}

// the per-thread kernels keep a replicate's values in arrays of KMAX = 8, 32 or 256 entries, the smallest that holds
// the largest K: launch(std::integral_constant<int, KMAX>)
template <class Launch>
static void with_kmax(int k, Launch launch) {
    if (k <= 8)
        launch(std::integral_constant<int, 8>());
    else if (k <= 32)
        launch(std::integral_constant<int, 32>());
    else
        launch(std::integral_constant<int, 256>());
}

template <int AMAX>
static void launch_fit(int kmax, const int *vals, const double *cdf, const int *cnt, const int *K, const int *n,
                       const int *status, const int *A, int n_loci, int kcap, int S, const AlleleParams &P, double *rm,
                       double *rw, double *rs, unsigned char *rp, cudaStream_t st) {
    const unsigned grid = (unsigned)(((long long)n_loci * P.num_bootstrap + 127) / 128);
    with_kmax(kmax, [&](auto km) {
        alleles_fit_kernel<decltype(km)::value, AMAX><<<grid, 128, 0, st>>>(vals, cdf, cnt, K, n, status, A, n_loci, kcap,
                                                                             S, P, rm, rw, rs, rp);
    });
}

// strk_call_alleles (n_alleles = the batch-wide count, A_loc = NULL) and strk_call_alleles_ploidy (A_loc = per-locus
// counts 1..ALL_MAX_ALLELES, n_alleles = 0): output rows and replicate scratch have S = the largest count of the batch
static int call_alleles_impl(const char *fn, strk_ctx *ctx, const int32_t *cn, const double *weights,
                             const int64_t *read_begin, int64_t n_loci, int n_alleles, const int32_t *A_loc,
                             int num_bootstrap, int min_reads, int min_allele_reads, int force_gm_filter,
                             double expansion_ratio, int filter_factor, int n_init, uint64_t seed, int32_t *out_i,
                             double *out_d, int32_t *out_status, double *ms_out) {
    if (!ctx || !read_begin || !out_i || !out_d || !out_status) return set_err(STRK_ERR_ARG, "%s: null argument", fn);
    if (n_loci < 0 || n_loci > 0x7fffffffLL / 4096) return set_err(STRK_ERR_ARG, "%s: bad locus count", fn);
    AlleleParams P;
    int rc = alleles_params(&P, n_alleles, A_loc != nullptr, num_bootstrap, min_reads, min_allele_reads, force_gm_filter,
                            expansion_ratio, filter_factor, n_init, seed);
    if (rc) return rc;
    if (n_loci == 0) return STRK_OK;
    int S = n_alleles;
    if (A_loc) {
        for (int64_t l = 0; l < n_loci; ++l) {
            if (A_loc[l] < 1 || A_loc[l] > ALL_MAX_ALLELES)
                return set_err(STRK_ERR_UNSUPPORTED, "%s: locus %lld has n_alleles = %d (1 to %d are implemented)", fn,
                               (long long)l, A_loc[l], ALL_MAX_ALLELES);
            S = std::max(S, (int)A_loc[l]);
        }
    }
    const int64_t n_reads = read_begin[n_loci];
    if (read_begin[0] != 0 || n_reads < 0 || (n_reads && (!cn || !weights)))
        return set_err(STRK_ERR_ARG, "%s: read_begin must run from 0 to the number of reads", fn);
    // shallow loci (<= ALL_SHALLOW_READS reads) set the stride of the per-locus arrays; deep ones are listed with
    // ragged offsets of min(reads, ALL_DEEP_MAX_K) entries
    int max_n = 1;
    std::vector<int> deep;
    std::vector<long long> doff(1, 0);
    for (int64_t l = 0; l < n_loci; ++l) {
        const int64_t d = read_begin[l + 1] - read_begin[l];
        if (d < 0) return set_err(STRK_ERR_ARG, "%s: locus %lld has a non-monotone read_begin", fn, (long long)l);
        if (d > 0x7fffffffLL) return set_err(STRK_ERR_UNSUPPORTED, "%s: locus %lld has %lld reads", fn, (long long)l, (long long)d);
        if (d > ALL_SHALLOW_READS) {
            deep.push_back((int)l);
            doff.push_back(doff.back() + std::min<int64_t>(d, ALL_DEEP_MAX_K));
        } else if (d > max_n) {
            max_n = (int)d;
        }
    }
    const int n_deep = (int)deep.size();
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int kcap = max_n, B = num_bootstrap;
    // context-owned buffers, recycled across calls (no cudaMalloc / cudaFree in the steady state)
    cudaError_t e = cudaSuccess;
    auto take_i = [&](int slot, size_t n) -> int * {
        if (e == cudaSuccess) e = ctx->al_i[slot].reserve(n ? n : 1);
        return ctx->al_i[slot].p;
    };
    auto take_d = [&](int slot, size_t n) -> double * {
        if (e == cudaSuccess) e = ctx->al_d[slot].reserve(n ? n : 1);
        return ctx->al_d[slot].p;
    };
    int *d_cn = take_i(0, (size_t)n_reads), *d_vals = take_i(1, (size_t)n_loci * kcap);
    int *d_cnt = take_i(2, (size_t)n_loci * kcap), *d_K = take_i(3, (size_t)n_loci), *d_n = take_i(4, (size_t)n_loci);
    int *d_status = take_i(5, (size_t)n_loci), *d_kmax = take_i(6, 1), *d_oi = take_i(7, (size_t)n_loci * (1 + 5 * S));
    int *d_A = A_loc ? take_i(8, (size_t)n_loci) : nullptr;
    double *d_w = take_d(0, (size_t)n_reads), *d_cdf = take_d(1, (size_t)n_loci * kcap);
    double *d_od = take_d(2, (size_t)n_loci * 3 * S);
    int *d_deep = take_i(9, (size_t)n_deep), *d_dvals = take_i(10, (size_t)doff.back()), *d_dK = take_i(11, (size_t)n_deep);
    double *d_dcdf = take_d(3, (size_t)doff.back());
    if (e == cudaSuccess) e = ctx->al_rb.reserve((size_t)n_loci + 1);
    if (e == cudaSuccess) e = ctx->al_doff.reserve((size_t)n_deep + 1);
    long long *d_rb = ctx->al_rb.p, *d_doff = ctx->al_doff.p;
    if (e == cudaSuccess && n_reads) e = cudaMemcpyAsync(d_cn, cn, (size_t)n_reads * sizeof(int), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && n_reads) e = cudaMemcpyAsync(d_w, weights, (size_t)n_reads * sizeof(double), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(d_rb, read_begin, ((size_t)n_loci + 1) * sizeof(long long), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && d_A) e = cudaMemcpyAsync(d_A, A_loc, (size_t)n_loci * sizeof(int), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && n_deep)
        e = cudaMemcpyAsync(d_deep, deep.data(), (size_t)n_deep * sizeof(int), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && n_deep)
        e = cudaMemcpyAsync(d_doff, doff.data(), ((size_t)n_deep + 1) * sizeof(long long), cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(STRK_ERR_NOMEM, "%s: %s", fn, cudaGetErrorString(e));
    }
    cudaEvent_t e0, e1;
    e0 = ctx->ev[0], e1 = ctx->ev[1];  // context-owned: nothing to release on an error path
    CU(cudaEventRecord(e0, st));
    CU(cudaMemsetAsync(d_kmax, 0, sizeof(int), st));
    alleles_prepare_kernel<<<(unsigned)((n_loci + 127) / 128), 128, 0, st>>>(d_cn, d_w, d_rb, d_A, (int)n_loci, min_reads,
                                                                             kcap, d_vals, d_cdf, d_cnt, d_K, d_n,
                                                                             d_status, d_kmax);
    CU(cudaGetLastError());
    std::vector<int> deep_K((size_t)n_deep);
    if (n_deep) {
        const size_t prep_smem = ALL_DEEP_TABLE * sizeof(unsigned long long) + ALL_DEEP_MAX_K * sizeof(int);
        CU(smem_opt_in(alleles_deep_prepare_kernel, prep_smem));
        alleles_deep_prepare_kernel<<<(unsigned)n_deep, 256, prep_smem, st>>>(d_cn, d_w, d_rb, d_deep, d_doff, min_reads,
                                                                             kcap, d_dvals, d_dcdf, d_K, d_dK, d_status,
                                                                             d_vals);
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(deep_K.data(), d_dK, (size_t)n_deep * sizeof(int), cudaMemcpyDeviceToHost, st));
    }
    int kmax = 0;
    CU(cudaMemcpyAsync(&kmax, d_kmax, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (int d = 0; d < n_deep; ++d)
        if (deep_K[d] > ALL_DEEP_MAX_K)
            return set_err(STRK_ERR_UNSUPPORTED, "%s: locus %d has more than %d distinct copy numbers", fn, deep[d],
                           ALL_DEEP_MAX_K);
    // replicate estimates, in chunks of loci that keep the scratch near 256 MB (context-owned, recycled across calls)
    const size_t per_locus = (size_t)S * B * 3 * sizeof(double) + (size_t)B;
    int64_t chunk = (int64_t)((size_t)1 << 28) / (int64_t)per_locus;
    if (chunk < 1) chunk = 1;
    if (chunk > n_loci) chunk = n_loci;
    for (int k = 0; k < 3 && e == cudaSuccess; ++k) e = ctx->al_rep[k].reserve((size_t)chunk * S * B);
    if (e == cudaSuccess) e = ctx->al_peaks.reserve((size_t)chunk * B);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(STRK_ERR_NOMEM, "%s: %s", fn, cudaGetErrorString(e));
    }
    double *rm = ctx->al_rep[0].p, *rw = ctx->al_rep[1].p, *rs = ctx->al_rep[2].p;
    unsigned char *rp = ctx->al_peaks.p;
    int np2 = 1;
    while (np2 < B) np2 <<= 1;
    const size_t agg_smem = (size_t)np2 * (sizeof(double) + sizeof(int));
    CU(smem_opt_in(alleles_aggregate_kernel, agg_smem));
    for (int64_t l0 = 0; l0 < n_loci; l0 += chunk) {
        const int nl = (int)std::min<int64_t>(chunk, n_loci - l0);
        const int *v = d_vals + (size_t)l0 * kcap, *c = d_cnt + (size_t)l0 * kcap;
        const double *p = d_cdf + (size_t)l0 * kcap;
        AlleleParams Pc = P;
        Pc.seed = seed + 0x9E3779B97F4A7C15ull * (unsigned long long)(l0 / chunk);  // distinct streams per chunk
        const int *a = d_A ? d_A + l0 : nullptr;
        if (S <= 2)  // the two-component code only
            launch_fit<2>(kmax, v, p, c, d_K + l0, d_n + l0, d_status + l0, a, nl, kcap, S, Pc, rm, rw, rs, rp, st);
        else
            launch_fit<ALL_MAX_ALLELES>(kmax, v, p, c, d_K + l0, d_n + l0, d_status + l0, a, nl, kcap, S, Pc, rm, rw, rs,
                                        rp, st);
        CU(cudaGetLastError());
        const int d0 = (int)(std::lower_bound(deep.begin(), deep.end(), (int)l0) - deep.begin());
        const int d1 = (int)(std::lower_bound(deep.begin(), deep.end(), (int)(l0 + nl)) - deep.begin());
        if (d1 > d0) {
            // every (deep locus, replicate) a warp; shared memory sized by the chunk's largest deep K
            const int kd = *std::max_element(deep_K.begin() + d0, deep_K.begin() + d1);
            const size_t fit_smem = (size_t)kd * (sizeof(double) * (1 + ALL_DEEP_WARPS) + sizeof(int) * ALL_DEEP_WARPS);
            CU(smem_opt_in(alleles_deep_fit_kernel, fit_smem));
            const dim3 grid((unsigned)(d1 - d0), (unsigned)((B + ALL_DEEP_WARPS - 1) / ALL_DEEP_WARPS));
            alleles_deep_fit_kernel<<<grid, 32 * ALL_DEEP_WARPS, fit_smem, st>>>(d_deep + d0, d_doff + d0, d_dvals, d_dcdf,
                                                                               d_K, d_n, d_status, d_A, (int)l0, S, P,
                                                                               rm, rw, rs, rp);
            CU(cudaGetLastError());
        }
        alleles_aggregate_kernel<<<(unsigned)nl, 256, agg_smem, st>>>(rm, rw, rs, rp, d_status + l0, v, kcap, nl, a, S, B,
                                                                      d_oi + (size_t)l0 * (1 + 5 * S),
                                                                      d_od + (size_t)l0 * 3 * S);
        CU(cudaGetLastError());
    }
    CU(cudaEventRecord(e1, st));
    CU(cudaMemcpyAsync(out_i, d_oi, (size_t)n_loci * (1 + 5 * S) * sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(out_d, d_od, (size_t)n_loci * 3 * S * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(out_status, d_status, (size_t)n_loci * sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (ms_out) {
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, e0, e1));
        *ms_out = (double)ms;
    }
    return STRK_OK;
}

extern "C" int strk_call_alleles(strk_ctx *ctx, const int32_t *cn, const double *weights, const int64_t *read_begin,
                                 int64_t n_loci, int n_alleles, int num_bootstrap, int min_reads, int min_allele_reads,
                                 int force_gm_filter, double expansion_ratio, int filter_factor, int n_init,
                                 uint64_t seed, int32_t *out_i, double *out_d, int32_t *out_status, double *ms_out) {
    return call_alleles_impl("strk_call_alleles", ctx, cn, weights, read_begin, n_loci, n_alleles, nullptr, num_bootstrap,
                             min_reads, min_allele_reads, force_gm_filter, expansion_ratio, filter_factor, n_init, seed,
                             out_i, out_d, out_status, ms_out);
}

extern "C" int strk_call_alleles_ploidy(strk_ctx *ctx, const int32_t *cn, const double *weights,
                                        const int64_t *read_begin, int64_t n_loci, const int32_t *n_alleles,
                                        int num_bootstrap, int min_reads, int min_allele_reads, int force_gm_filter,
                                        double expansion_ratio, int filter_factor, int n_init, uint64_t seed,
                                        int32_t *out_i, double *out_d, int32_t *out_status, double *ms_out) {
    if (!n_alleles && n_loci > 0) return set_err(STRK_ERR_ARG, "strk_call_alleles_ploidy: null argument");
    return call_alleles_impl("strk_call_alleles_ploidy", ctx, cn, weights, read_begin, n_loci, 0, n_alleles,
                             num_bootstrap, min_reads, min_allele_reads, force_gm_filter, expansion_ratio, filter_factor,
                             n_init, seed, out_i, out_d, out_status, ms_out);
}

extern "C" int strk_gmm_fit_counts(strk_ctx *ctx, const double *x, const int32_t *counts, const int32_t *K,
                                   const int32_t *init, int64_t n_problems, int kcap, int n_alleles, int num_bootstrap,
                                   int min_allele_reads, int force_gm_filter, double expansion_ratio, int filter_factor,
                                   int n_init, double *out) {
    if (!ctx || !x || !counts || !K || !init || !out) return set_err(STRK_ERR_ARG, "strk_gmm_fit_counts: null argument");
    if (n_problems < 0 || n_problems > 0x7fffffff || kcap < 1 || kcap > 256)
        return set_err(STRK_ERR_ARG, "strk_gmm_fit_counts: bad sizes");
    AlleleParams P;
    int rc = alleles_params(&P, n_alleles, false, num_bootstrap, 0, min_allele_reads, force_gm_filter, expansion_ratio,
                            filter_factor, n_init, 0);
    if (rc) return rc;
    if (n_problems == 0) return STRK_OK;
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    TmpDev dev{st};
    double *d_x = nullptr, *d_out = nullptr;
    int *d_c = nullptr, *d_K = nullptr, *d_init = nullptr;
    cudaError_t e = dev.up(&d_x, x, (size_t)n_problems * kcap);
    if (e == cudaSuccess) e = dev.up(&d_c, (const int *)counts, (size_t)n_problems * kcap);
    if (e == cudaSuccess) e = dev.up(&d_K, (const int *)K, (size_t)n_problems);
    if (e == cudaSuccess) e = dev.up(&d_init, (const int *)init, (size_t)n_problems * 2 * n_init);
    if (e == cudaSuccess) e = dev.get(&d_out, (size_t)n_problems * 7);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(STRK_ERR_NOMEM, "strk_gmm_fit_counts: %s", cudaGetErrorString(e));
    }
    for (int64_t q = 0; q < n_problems; ++q)
        if (K[q] < 1 || K[q] > kcap) return set_err(STRK_ERR_ARG, "strk_gmm_fit_counts: problem %lld has K = %d", (long long)q, K[q]);
    const unsigned grid = (unsigned)((n_problems + 127) / 128);
    with_kmax(kcap, [&](auto km) {
        gmm_fit_counts_kernel<decltype(km)::value><<<grid, 128, 0, st>>>(d_x, d_c, d_K, d_init, (int)n_problems, kcap, P,
                                                                         d_out);
    });
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out, d_out, (size_t)n_problems * 7 * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return STRK_OK;
}

// strk_gmm_fit_counts_ploidy (per-thread fit, kcap <= 256) and strk_gmm_fit_counts_deep (warp fit of deep loci,
// kcap <= ALL_DEEP_MAX_K): the same arguments, checks and output
static int gmm_fit_counts_impl(const char *fn, bool deep, strk_ctx *ctx, const double *x, const int32_t *counts,
                               const int32_t *K, const int32_t *n_alleles, const int32_t *init, int64_t n_problems,
                               int kcap, int num_bootstrap, int min_allele_reads, int force_gm_filter,
                               double expansion_ratio, int filter_factor, int n_init, uint64_t seed, double *out) {
    if (!ctx || !x || !counts || !K || !n_alleles || !out) return set_err(STRK_ERR_ARG, "%s: null argument", fn);
    if (n_problems < 0 || n_problems > 0x7fffffff || kcap < 1 || kcap > (deep ? ALL_DEEP_MAX_K : 256))
        return set_err(STRK_ERR_ARG, "%s: bad sizes", fn);
    AlleleParams P;
    int rc = alleles_params(&P, 0, true, num_bootstrap, 0, min_allele_reads, force_gm_filter, expansion_ratio,
                            filter_factor, n_init, seed);
    if (rc) return rc;
    if (n_problems == 0) return STRK_OK;
    // seeds of problem q: for nc = A, A-1, ..., 2, n_init rows of nc indices, problems back to back
    std::vector<long long> off((size_t)n_problems + 1, 0);
    int S = 1;
    for (int64_t q = 0; q < n_problems; ++q) {
        const int A = n_alleles[q];
        if (A < 1 || A > ALL_MAX_ALLELES)
            return set_err(STRK_ERR_UNSUPPORTED, "%s: problem %lld has n_alleles = %d (1 to %d are implemented)", fn,
                           (long long)q, A, ALL_MAX_ALLELES);
        if (K[q] < 1 || K[q] > kcap) return set_err(STRK_ERR_ARG, "%s: problem %lld has K = %d", fn, (long long)q, K[q]);
        int n = 0, distinct = 0;
        for (int j = 0; j < K[q]; ++j) {
            const int cj = counts[(size_t)q * kcap + j];
            if (cj < 0) return set_err(STRK_ERR_ARG, "%s: problem %lld has a negative count", fn, (long long)q);
            n += cj, distinct += cj > 0;
        }
        if (n < 1 || (distinct > 1 && n < A))
            return set_err(STRK_ERR_ARG, "%s: problem %lld has %d points for %d components", fn, (long long)q, n, A);
        S = std::max(S, A);
        off[q + 1] = off[q] + (long long)n_init * (A * (A + 1) / 2 - 1);
    }
    if (init)
        for (int64_t q = 0; q < n_problems; ++q)
            for (long long i = off[q]; i < off[q + 1]; ++i)
                if (init[i] < 0 || init[i] >= K[q])
                    return set_err(STRK_ERR_ARG, "%s: problem %lld has a seed index %d outside 0..%d", fn, (long long)q,
                                   init[i], K[q] - 1);
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    TmpDev dev{st};
    double *d_x = nullptr, *d_out = nullptr;
    int *d_c = nullptr, *d_K = nullptr, *d_A = nullptr, *d_init = nullptr;
    long long *d_off = nullptr;
    cudaError_t e = dev.up(&d_x, x, (size_t)n_problems * kcap);
    if (e == cudaSuccess) e = dev.up(&d_c, (const int *)counts, (size_t)n_problems * kcap);
    if (e == cudaSuccess) e = dev.up(&d_K, (const int *)K, (size_t)n_problems);
    if (e == cudaSuccess) e = dev.up(&d_A, (const int *)n_alleles, (size_t)n_problems);
    if (e == cudaSuccess && init) e = dev.up(&d_init, (const int *)init, (size_t)off[n_problems]);
    if (e == cudaSuccess && init) e = dev.up(&d_off, off.data(), (size_t)n_problems);
    if (e == cudaSuccess) e = dev.get(&d_out, (size_t)n_problems * (3 * S + 1));
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(STRK_ERR_NOMEM, "%s: %s", fn, cudaGetErrorString(e));
    }
    if (deep) {
        const size_t smem = (size_t)kcap * (sizeof(double) + sizeof(int)) * ALL_DEEP_WARPS;
        CU(smem_opt_in(gmm_fit_counts_deep_kernel, smem));
        gmm_fit_counts_deep_kernel<<<(unsigned)((n_problems + ALL_DEEP_WARPS - 1) / ALL_DEEP_WARPS), 32 * ALL_DEEP_WARPS,
                                     smem, st>>>(d_x, d_c, d_K, d_A, d_init, d_off, (int)n_problems, kcap, S, P, d_out);
    } else {
        const unsigned grid = (unsigned)((n_problems + 127) / 128);
        with_kmax(kcap, [&](auto km) {
            gmm_fit_counts_ploidy_kernel<decltype(km)::value><<<grid, 128, 0, st>>>(d_x, d_c, d_K, d_A, d_init, d_off,
                                                                                    (int)n_problems, kcap, S, P, d_out);
        });
    }
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out, d_out, (size_t)n_problems * (3 * S + 1) * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return STRK_OK;
}

extern "C" int strk_gmm_fit_counts_ploidy(strk_ctx *ctx, const double *x, const int32_t *counts, const int32_t *K,
                                          const int32_t *n_alleles, const int32_t *init, int64_t n_problems, int kcap,
                                          int num_bootstrap, int min_allele_reads, int force_gm_filter,
                                          double expansion_ratio, int filter_factor, int n_init, uint64_t seed,
                                          double *out) {
    return gmm_fit_counts_impl("strk_gmm_fit_counts_ploidy", false, ctx, x, counts, K, n_alleles, init, n_problems, kcap,
                               num_bootstrap, min_allele_reads, force_gm_filter, expansion_ratio, filter_factor, n_init,
                               seed, out);
}

extern "C" int strk_gmm_fit_counts_deep(strk_ctx *ctx, const double *x, const int32_t *counts, const int32_t *K,
                                        const int32_t *n_alleles, const int32_t *init, int64_t n_problems, int kcap,
                                        int num_bootstrap, int min_allele_reads, int force_gm_filter,
                                        double expansion_ratio, int filter_factor, int n_init, uint64_t seed,
                                        double *out) {
    return gmm_fit_counts_impl("strk_gmm_fit_counts_deep", true, ctx, x, counts, K, n_alleles, init, n_problems, kcap,
                               num_bootstrap, min_allele_reads, force_gm_filter, expansion_ratio, filter_factor, n_init,
                               seed, out);
}

extern "C" int strk_alleles_aggregate(strk_ctx *ctx, const double *rep_means, const double *rep_weights,
                                      const double *rep_stdevs, const uint8_t *rep_peaks, int64_t n_loci, int n_alleles,
                                      int num_bootstrap, int32_t *out_i, double *out_d) {
    if (!ctx || !rep_means || !rep_weights || !rep_stdevs || !rep_peaks || !out_i || !out_d)
        return set_err(STRK_ERR_ARG, "strk_alleles_aggregate: null argument");
    if (n_alleles < 1 || n_alleles > ALL_MAX_ALLELES || num_bootstrap < 1 || num_bootstrap > ALL_MAX_BOOT || n_loci < 0 ||
        n_loci > 0x7fffffff)
        return set_err(STRK_ERR_ARG, "strk_alleles_aggregate: bad sizes");
    if (n_loci == 0) return STRK_OK;
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int A = n_alleles, B = num_bootstrap;
    TmpDev dev{st};
    double *rm = nullptr, *rw = nullptr, *rs = nullptr, *d_od = nullptr;
    unsigned char *rp = nullptr;
    int *d_status = nullptr, *d_oi = nullptr;
    const size_t nrep = (size_t)n_loci * A * B;
    cudaError_t e = dev.up(&rm, rep_means, nrep);
    if (e == cudaSuccess) e = dev.up(&rw, rep_weights, nrep);
    if (e == cudaSuccess) e = dev.up(&rs, rep_stdevs, nrep);
    if (e == cudaSuccess) e = dev.up(&rp, (const unsigned char *)rep_peaks, (size_t)n_loci * B);
    if (e == cudaSuccess) e = dev.get(&d_status, (size_t)n_loci);
    if (e == cudaSuccess) e = dev.get(&d_oi, (size_t)n_loci * (1 + 5 * A));
    if (e == cudaSuccess) e = dev.get(&d_od, (size_t)n_loci * 3 * A);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(STRK_ERR_NOMEM, "strk_alleles_aggregate: %s", cudaGetErrorString(e));
    }
    CU(cudaMemsetAsync(d_status, 0, (size_t)n_loci * sizeof(int), st));
    int np2 = 1;
    while (np2 < B) np2 <<= 1;
    const size_t agg_smem = (size_t)np2 * (sizeof(double) + sizeof(int));
    CU(smem_opt_in(alleles_aggregate_kernel, agg_smem));
    alleles_aggregate_kernel<<<(unsigned)n_loci, 256, agg_smem, st>>>(rm, rw, rs, rp, d_status, nullptr, 1, (int)n_loci,
                                                                      nullptr, A, B, d_oi, d_od);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out_i, d_oi, (size_t)n_loci * (1 + 5 * A) * sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(out_d, d_od, (size_t)n_loci * 3 * A * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return STRK_OK;
}
