// alleles.cuh -- bootstrap resampling + Gaussian-mixture allele calling, batched over loci (SURVEY 8f N3).
//
// Follows the reference's call_alleles (strkit/call/allele.py:176-336) with its helpers
// get_resampled_bootstrapped_reads (:126-173, the separate_strands=False branch both call sites use,
// call_locus.py:201-214,255-268), fit_gmm (:56-123), make_single_gaussian / GMMParams.make_fitted_gmm
// (strkit/call/gmm.py:59-80) and, underneath, scikit-learn 1.9.0's GaussianMixture (spherical, k-means++
// init, n_init restarts, tol 1e-3, max_iter 100, reg_covar 1e-6) restated in float64:
//
//   alleles_prepare_kernel   one thread per locus: distinct copy numbers, their resampling probabilities
//   alleles_fit_kernel       one thread per (locus, bootstrap replicate): multinomial resample (counter-based
//                            Philox RNG), k-means++ seeding, EM, the reference's peak filters
//   alleles_aggregate_kernel one CTA per locus: per-allele stable sort of the replicate estimates,
//                            interpolated-inverted-CDF percentiles, median, modal peak count
//
// The allele count A belongs to the locus (STRkitLocus.n_alleles, set by the ploidy config), 1..ALL_MAX_ALLELES.
// A <= 2 runs the two-component code (fit_replicate); A >= 3 runs fit_gmm's staged loop over k components
// (fit_replicate_k): k-means++ for k centres, EM with k components, refits with fewer components while the
// filters find useless ones, and the reference's random fill of the alleles a replicate has no peak for.
//
// A bootstrap replicate of integer copy numbers is a multiset over the locus' K distinct values, so it is
// carried as K counts; EM on (value, count) pairs is the same arithmetic as EM on the expanded sample
// (identical points have identical responsibilities).  Random streams differ from numpy's / sklearn's, so
// results agree with the reference statistically, not bit for bit; the deterministic parts (EM given the
// seeds, the aggregation) are tested exactly.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define ALL_MAX_BOOT 4096   // replicates per locus the aggregation kernel sorts in shared memory
#define ALL_N_INIT_MAX 8
#define ALL_MAX_ALLELES 8   // components per locus (fit_replicate_k keeps its arrays this wide)
#define ALL_SHALLOW_READS 256  // loci with more reads are deep: alleles_deep_prepare_kernel / alleles_deep_fit_kernel
#define ALL_DEEP_MAX_K 4096    // distinct copy numbers of a deep locus (bounds the deep fit's shared memory)
#define ALL_DEEP_WARPS 4       // warps per CTA of the deep fit, one (locus, replicate) each
#define ALL_DEEP_STREAM 0x80000000u  // replicate-word bit of deep streams: shallow replicates are < ALL_MAX_BOOT

struct AlleleParams {
    int n_alleles;          // 1 or 2: the batch-wide count of strk_call_alleles (per-locus counts come as an array)
    int num_bootstrap;
    int min_reads;
    int n_init;             // GMMParams.n_init (params.py:166-172: 3)
    int max_iter;           // sklearn default 100
    int force_gm_filter;
    double tol;             // sklearn default 1e-3
    double reg_covar;       // sklearn default 1e-6
    double allele_filter;   // (min_allele_reads - 0.1) / num_bootstrap  (allele.py:243: concat_samples.shape[0])
    double expansion_ratio; // params.gm_filter_expansion_ratio
    double filter_weight;   // 1 / (filter_factor * 2)
    int filter_factor;      // the k-component filter's threshold is 1 / (filter_factor * k)
    double small_allele_min;  // allele.py:47
    unsigned long long seed;
};

// ---------------------------------------------------------------------------------------------- RNG
struct Philox {
    uint32_t key0, key1, c0, c1, c2, c3;
    uint32_t out[4];
    int have;
    __device__ __forceinline__ void init(unsigned long long seed, uint32_t a, uint32_t b) {
        key0 = (uint32_t)seed;
        key1 = (uint32_t)(seed >> 32);
        c0 = 0;
        c1 = 0;
        c2 = a;
        c3 = b;
        have = 0;
    }
    // jump to counter (lo, hi): the next two uniforms are the pair of that counter
    __device__ __forceinline__ void seek(uint32_t lo, uint32_t hi) {
        c0 = lo;
        c1 = hi;
        have = 0;
    }
    __device__ __forceinline__ void round(uint32_t &x0, uint32_t &x1, uint32_t &x2, uint32_t &x3, uint32_t k0,
                                          uint32_t k1) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, x0), lo0 = 0xD2511F53u * x0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, x2), lo1 = 0xCD9E8D57u * x2;
        const uint32_t y0 = hi1 ^ x1 ^ k0, y1 = lo1, y2 = hi0 ^ x3 ^ k1, y3 = lo0;
        x0 = y0, x1 = y1, x2 = y2, x3 = y3;
    }
    __device__ __forceinline__ void refill() {
        uint32_t x0 = c0, x1 = c1, x2 = c2, x3 = c3, k0 = key0, k1 = key1;
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            round(x0, x1, x2, x3, k0, k1);
            k0 += 0x9E3779B9u;
            k1 += 0xBB67AE85u;
        }
        out[0] = x0, out[1] = x1, out[2] = x2, out[3] = x3;
        if (++c0 == 0) ++c1;
        have = 4;
    }
    // uniform double in [0, 1), 53 bits
    __device__ __forceinline__ double uniform() {
        if (have < 2) refill();
        const uint32_t a = out[have - 1], b = out[have - 2];
        have -= 2;
        const unsigned long long u = ((unsigned long long)a << 32) | b;
        return (double)(u >> 11) * (1.0 / 9007199254740992.0);
    }
};

// ---------------------------------------------------------------------------------------------- prepare
// status: 0 = bootstrap + GMM, 1 = fewer than min_reads reads (reference returns None, allele.py:192-193),
//         2 = a single distinct value (no bootstrap, allele.py:196-214),
//         3 = fewer reads than the locus' allele count A (A_arr; NULL = no per-locus count): every replicate with
//             two distinct values would reach GaussianMixture(A).fit on fewer than A samples, which raises
__global__ void alleles_prepare_kernel(const int *__restrict__ cn, const double *__restrict__ w,
                                       const long long *__restrict__ read_begin, const int *__restrict__ A_arr,
                                       int n_loci, int min_reads, int kcap,
                                       int *__restrict__ vals, double *__restrict__ cdf, int *__restrict__ cnt,
                                       int *__restrict__ K_out,
                                       int *__restrict__ n_out, int *__restrict__ status, int *__restrict__ k_max) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= n_loci) return;
    const long long r0 = read_begin[l], r1 = read_begin[l + 1];
    const int n = (int)(r1 - r0);
    n_out[l] = n;
    if (n > ALL_SHALLOW_READS) return;  // deep: alleles_deep_prepare_kernel
    int *v = vals + (size_t)l * kcap;
    double *p = cdf + (size_t)l * kcap;
    int *q = cnt + (size_t)l * kcap;
    int K = 0;
    // insertion into a sorted list of distinct values, probabilities and read counts accumulated per value
    // (kcap >= the longest locus of the batch, so the list cannot overflow)
    for (long long r = r0; r < r1; ++r) {
        const int x = cn[r];
        const double wx = w[r];
        int lo = 0;
        while (lo < K && v[lo] < x) ++lo;
        if (lo < K && v[lo] == x) {
            p[lo] += wx;
            q[lo] += 1;
        } else if (K < kcap) {
            for (int j = K; j > lo; --j) v[j] = v[j - 1], p[j] = p[j - 1], q[j] = q[j - 1];
            v[lo] = x;
            p[lo] = wx;
            q[lo] = 1;
            ++K;
        }
    }
    // cumulative, normalised by the total like numpy's Generator.choice (cdf /= cdf[-1])
    double acc = 0.0;
    for (int j = 0; j < K; ++j) {
        acc += p[j];
        p[j] = acc;
    }
    for (int j = 0; j < K; ++j) p[j] /= acc;
    K_out[l] = K;
    status[l] = n < min_reads ? 1 : (K == 1 ? 2 : (A_arr && n < A_arr[l] ? 3 : 0));
    atomicMax(k_max, K);
}

// ---------------------------------------------------------------------------------------------- GMM
struct Gmm2 {
    double mean[2], cov[2], weight[2];
    int n_comp;
};

// sklearn _estimate_log_gaussian_prob (spherical, one feature) + log weight of one component, for one x
__device__ __forceinline__ double gmm_wlp1(double x, double mean, double pchol, double logw) {
    // separately rounded products and sums, in sklearn's order: the three terms cancel almost completely for
    // a point near the mean (precision up to 1e6), so a fused multiply-add here would change the low bits
    const double prec = __dmul_rn(pchol, pchol);
    const double t1 = __dmul_rn(__dmul_rn(mean, mean), prec);
    const double t2 = __dmul_rn(2.0, __dmul_rn(__dmul_rn(x, mean), prec));
    const double t3 = __dmul_rn(__dmul_rn(x, x), prec);
    const double lp = __dadd_rn(__dsub_rn(t1, t2), t3);
    return __dadd_rn(__dadd_rn(__dmul_rn(-0.5, __dadd_rn(1.8378770664093453, lp)), log(pchol)), logw);
}

__device__ __forceinline__ void gmm_wlp(double x, const double mean[2], const double pchol[2], const double logw[2],
                                        double out[2]) {
#pragma unroll
    for (int k = 0; k < 2; ++k) out[k] = gmm_wlp1(x, mean[k], pchol[k], logw[k]);
}

// EM from the k-means++ seeds (value indices i0, i1): GaussianMixture._initialize with one-hot responsibilities on
// the two seed points, then e-step / m-step until |change of the lower bound| < tol (sklearn BaseMixture.fit_predict).
template <int KMAX>
__device__ double gmm_em(const double *x, const int *c, int K, int n, int i0, int i1, const AlleleParams &P, Gmm2 &g,
                         int *n_iter_out) {
    const double eps10 = 10.0 * 2.220446049250313e-16;
    double mean[2], cov[2], weight[2], pchol[2], logw[2];
    {
        const int idx[2] = {i0, i1};
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const double nk = 1.0 + eps10, xv = x[idx[k]];
            mean[k] = xv / nk;
            cov[k] = __dadd_rn(__dsub_rn(__ddiv_rn(__dmul_rn(xv, xv), nk), __dmul_rn(mean[k], mean[k])), P.reg_covar);
            weight[k] = nk / (double)n;
            pchol[k] = 1.0 / sqrt(cov[k]);
            logw[k] = log(weight[k]);
        }
    }
    double lower = -INFINITY;
    int it = 1;
    for (; it <= P.max_iter; ++it) {
        const double prev = lower;
        double nk[2] = {0.0, 0.0}, sx[2] = {0.0, 0.0}, sxx[2] = {0.0, 0.0}, ll = 0.0;
        for (int v = 0; v < K; ++v) {
            if (c[v] == 0) continue;
            double wl[2];
            gmm_wlp(x[v], mean, pchol, logw, wl);
            const double mx = fmax(wl[0], wl[1]);
            const double lse = mx + log(exp(wl[0] - mx) + exp(wl[1] - mx));
            const double cv = (double)c[v];
            ll += cv * lse;
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const double r = exp(wl[k] - lse) * cv;
                nk[k] += r;
                sx[k] += r * x[v];
                sxx[k] += r * x[v] * x[v];
            }
        }
        lower = ll / (double)n;
        double wsum = 0.0;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            nk[k] += eps10;
            mean[k] = sx[k] / nk[k];
            cov[k] = __dadd_rn(__dsub_rn(__ddiv_rn(sxx[k], nk[k]), __dmul_rn(mean[k], mean[k])), P.reg_covar);
            weight[k] = nk[k] / (double)n;
            wsum += weight[k];
        }
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            weight[k] /= wsum;
            // sklearn raises on cov <= 0 (ill-defined covariance); it cannot happen for integer data of this
            // range with reg_covar = 1e-6, the clamp only keeps the arithmetic finite
            pchol[k] = 1.0 / sqrt(cov[k] > 0.0 ? cov[k] : P.reg_covar);
            logw[k] = log(weight[k]);
        }
        if (fabs(lower - prev) < P.tol) break;
    }
    if (it > P.max_iter) it = P.max_iter;
#pragma unroll
    for (int k = 0; k < 2; ++k) g.mean[k] = mean[k], g.cov[k] = cov[k], g.weight[k] = weight[k];
    g.n_comp = 2;
    if (n_iter_out) *n_iter_out = it;
    return lower;
}

// sklearn.cluster.kmeans_plusplus for two centres on the (sorted) replicate: first centre uniform over the n points,
// second = the better of 2 + int(log 2) = 2 candidates drawn proportionally to the squared distance.
template <int KMAX>
__device__ void kmeanspp2(const double *x, const int *c, int K, int n, Philox &rng, int &i0, int &i1) {
    // first centre: point index floor(u * n) -> value index  (Generator-free restatement of RandomState.choice)
    {
        const double u = rng.uniform();
        long long pt = (long long)(u * (double)n);
        if (pt >= n) pt = n - 1;
        int v = 0;
        long long acc = 0;
        for (; v < K; ++v) {
            acc += c[v];
            if (pt < acc) break;
        }
        i0 = v < K ? v : K - 1;
    }
    double pot = 0.0;
    for (int v = 0; v < K; ++v) {
        const double d = x[v] - x[i0];
        pot += (double)c[v] * d * d;
    }
    double best_pot = INFINITY;
    int best = i0;
#pragma unroll 1
    for (int t = 0; t < 2; ++t) {
        const double r = rng.uniform() * pot;
        int v = 0;
        double acc = 0.0;
        int last_nonzero = 0;
        for (; v < K; ++v) {
            if (c[v]) last_nonzero = v;
            const double d = x[v] - x[i0];
            acc += (double)c[v] * d * d;
            if (c[v] && acc >= r) break;
        }
        const int cand = v < K ? v : last_nonzero;
        double cp = 0.0;
        for (int q = 0; q < K; ++q) {
            const double d0 = x[q] - x[i0], d1 = x[q] - x[cand];
            cp += (double)c[q] * fmin(d0 * d0, d1 * d1);
        }
        if (cp < best_pot) best_pot = cp, best = cand;
    }
    i1 = best;
}

// make_single_gaussian (gmm.py:72-80): mean and population variance of the replicate
__device__ __forceinline__ void single_gaussian(const double *x, const int *c, int K, int n, double &mean, double &var) {
    double s = 0.0;
    for (int v = 0; v < K; ++v) s += (double)c[v] * x[v];
    mean = s / (double)n;
    double q = 0.0;
    for (int v = 0; v < K; ++v) {
        const double d = x[v] - mean;
        q += (double)c[v] * d * d;
    }
    var = q / (double)n;
}

// fit_gmm's peak filters (allele.py:88-121) on a fitted 2-component model: number of useless components
__device__ __forceinline__ int gmm_useless(const Gmm2 &g, const AlleleParams &P) {
    const double lo = fmin(g.mean[0], g.mean[1]), hi = fmax(g.mean[0], g.mean[1]);
    const bool f2_strict = P.force_gm_filter || hi < P.expansion_ratio * fmax(lo, P.small_allele_min);
    const double thr2 = f2_strict ? P.filter_weight : 1.1920928955078125e-07;  // np.finfo(np.float32).eps
    int useless = 0;
#pragma unroll
    for (int k = 0; k < 2; ++k)
        if (!(g.weight[k] > P.allele_filter && g.weight[k] > thr2)) ++useless;
    return useless;
}

// One replicate -> the allele estimates the reference appends per bootstrap iteration (allele.py:249-293):
// out_m / out_w / out_s [n_alleles] sorted by mean, *n_peaks = g.means_.shape[0].
template <int KMAX>
__device__ void fit_replicate(const double *x, const int *c, int K, int n, int A, const AlleleParams &P, Philox &rng,
                              const int *forced_init, double *out_m, double *out_w, double *out_s, int *n_peaks) {
    int distinct = 0;
    for (int v = 0; v < K; ++v) distinct += c[v] != 0;
    bool single = distinct == 1 || A == 1;  // fit_gmm: len(mc) == 1, or n_components == 1
    Gmm2 best;
    if (!single) {
        double best_lb = -INFINITY;
        for (int t = 0; t < P.n_init; ++t) {
            int i0, i1;
            if (forced_init) {
                i0 = forced_init[2 * t];
                i1 = forced_init[2 * t + 1];
            } else {
                kmeanspp2<KMAX>(x, c, K, n, rng, i0, i1);
            }
            Gmm2 g;
            const double lb = gmm_em<KMAX>(x, c, K, n, i0, i1, P, g, nullptr);
            if (lb > best_lb || best_lb == -INFINITY) best_lb = lb, best = g;
        }
        // while n_components > 0: 2 -> (2 - n_useless); 1 -> single Gaussian; 0 -> the loop ends and g is returned
        const int useless = gmm_useless(best, P);
        if (useless == 1) single = true;
    }
    if (single) {
        double m, var;
        single_gaussian(x, c, K, n, m, var);
        const double s = sqrt(var);
        for (int a = 0; a < A; ++a) out_m[a] = m, out_w[a] = 1.0, out_s[a] = s;
        *n_peaks = 1;
    } else {
        const int first = best.mean[1] < best.mean[0] ? 1 : 0;  // stable argsort of two means
        out_m[0] = best.mean[first], out_w[0] = best.weight[first], out_s[0] = sqrt(best.cov[first]);
        out_m[1] = best.mean[1 - first], out_w[1] = best.weight[1 - first], out_s[1] = sqrt(best.cov[1 - first]);
        *n_peaks = 2;
    }
}

// ---------------------------------------------------------------------------------------------- k components
// fit_gmm for A >= 3 components (allele.py:56-123 over GaussianMixture(n_components = k)); the two-component code
// above stays the path of A <= 2, so those results do not depend on this one.
struct GmmK {
    double mean[ALL_MAX_ALLELES], cov[ALL_MAX_ALLELES], weight[ALL_MAX_ALLELES];
    int n_comp;
};

// EM from the seed value indices idx[0..NC): gmm_em with NC components, the same separately rounded products, the
// same init (one-hot responsibilities on the seed points + 10 eps: two components seeded on one point stay equal),
// a NC-way log-sum-exp and the same convergence rule.  NC is a template so the component arrays stay in registers.
template <int NC, int KMAX>
__device__ double gmm_em_k(const double *x, const int *c, int K, int n, const int *idx, const AlleleParams &P,
                           GmmK &g) {
    const double eps10 = 10.0 * 2.220446049250313e-16;
    double mean[NC], cov[NC], weight[NC], pchol[NC], logw[NC];
#pragma unroll
    for (int k = 0; k < NC; ++k) {
        const double nk = 1.0 + eps10, xv = x[idx[k]];
        mean[k] = xv / nk;
        cov[k] = __dadd_rn(__dsub_rn(__ddiv_rn(__dmul_rn(xv, xv), nk), __dmul_rn(mean[k], mean[k])), P.reg_covar);
        weight[k] = nk / (double)n;
        pchol[k] = 1.0 / sqrt(cov[k]);
        logw[k] = log(weight[k]);
    }
    double lower = -INFINITY;
    for (int it = 1; it <= P.max_iter; ++it) {
        const double prev = lower;
        double nk[NC], sx[NC], sxx[NC], ll = 0.0;
#pragma unroll
        for (int k = 0; k < NC; ++k) nk[k] = 0.0, sx[k] = 0.0, sxx[k] = 0.0;
        for (int v = 0; v < K; ++v) {
            if (c[v] == 0) continue;
            double wl[NC];
#pragma unroll
            for (int k = 0; k < NC; ++k) wl[k] = gmm_wlp1(x[v], mean[k], pchol[k], logw[k]);
            double mx = wl[0];
#pragma unroll
            for (int k = 1; k < NC; ++k) mx = fmax(mx, wl[k]);
            double se = 0.0;
#pragma unroll
            for (int k = 0; k < NC; ++k) se += exp(wl[k] - mx);
            const double lse = mx + log(se);
            const double cv = (double)c[v];
            ll += cv * lse;
#pragma unroll
            for (int k = 0; k < NC; ++k) {
                const double r = exp(wl[k] - lse) * cv;
                nk[k] += r;
                sx[k] += r * x[v];
                sxx[k] += r * x[v] * x[v];
            }
        }
        lower = ll / (double)n;
        double wsum = 0.0;
#pragma unroll
        for (int k = 0; k < NC; ++k) {
            nk[k] += eps10;
            mean[k] = sx[k] / nk[k];
            cov[k] = __dadd_rn(__dsub_rn(__ddiv_rn(sxx[k], nk[k]), __dmul_rn(mean[k], mean[k])), P.reg_covar);
            weight[k] = nk[k] / (double)n;
            wsum += weight[k];
        }
#pragma unroll
        for (int k = 0; k < NC; ++k) {
            weight[k] /= wsum;
            pchol[k] = 1.0 / sqrt(cov[k] > 0.0 ? cov[k] : P.reg_covar);
            logw[k] = log(weight[k]);
        }
        if (fabs(lower - prev) < P.tol) break;
    }
#pragma unroll
    for (int k = 0; k < NC; ++k) g.mean[k] = mean[k], g.cov[k] = cov[k], g.weight[k] = weight[k];
    g.n_comp = NC;
    return lower;
}

// sklearn _kmeans_plusplus (cluster/_kmeans.py:224-275) for k centres on the (value, count) pairs of a replicate:
// the first centre uniform over the n points; each further centre the best (first argmin of the potential) of
// 2 + int(log k) candidates drawn by searchsorted(cumsum(count * closest_dist_sq), u * pot, side="left"), clipped
// to the last point.  When every point already sits on a centre (pot = 0) every draw lands on point 0, the smallest
// value, and that centre is duplicated -- as scikit-learn does.
template <int KMAX>
__device__ void kmeanspp_k(const double *x, const int *c, int K, int n, int k, Philox &rng, int *idx) {
    {
        const double u = rng.uniform();
        long long pt = (long long)(u * (double)n);
        if (pt >= n) pt = n - 1;
        int v = 0;
        long long acc = 0;
        for (; v < K; ++v) {
            acc += c[v];
            if (pt < acc) break;
        }
        idx[0] = v < K ? v : K - 1;
    }
    double closest[KMAX];
    double pot = 0.0;
    for (int v = 0; v < K; ++v) {
        const double d = x[v] - x[idx[0]];
        closest[v] = d * d;
        pot += (double)c[v] * closest[v];
    }
    const int trials = 2 + (int)log((double)k);
    for (int ci = 1; ci < k; ++ci) {
        double best_pot = INFINITY;
        int best = 0;
#pragma unroll 1
        for (int t = 0; t < trials; ++t) {
            const double r = rng.uniform() * pot;
            int v = 0, last_nonzero = 0;
            double acc = 0.0;
            for (; v < K; ++v) {
                if (c[v]) last_nonzero = v;
                acc += (double)c[v] * closest[v];
                if (c[v] && acc >= r) break;
            }
            const int cand = v < K ? v : last_nonzero;
            double cp = 0.0;
            for (int q = 0; q < K; ++q) {
                const double d = x[q] - x[cand];
                cp += (double)c[q] * fmin(closest[q], d * d);
            }
            if (cp < best_pot) best_pot = cp, best = cand;
        }
        idx[ci] = best;
        pot = best_pot;
        for (int q = 0; q < K; ++q) {
            const double d = x[q] - x[best];
            closest[q] = fmin(closest[q], d * d);
        }
    }
}

// GaussianMixture(nc).fit: the best of n_init restarts (forced = n_init rows of nc seed indices, or NULL for k-means++)
template <int KMAX>
__device__ void gmm_fit_k(const double *x, const int *c, int K, int n, int nc, const AlleleParams &P, Philox &rng,
                          const int *forced, GmmK &best) {
    double best_lb = -INFINITY;
    for (int t = 0; t < P.n_init; ++t) {
        int idx[ALL_MAX_ALLELES];
        if (forced) {
            for (int j = 0; j < nc; ++j) idx[j] = forced[t * nc + j];
        } else {
            kmeanspp_k<KMAX>(x, c, K, n, nc, rng, idx);
        }
        GmmK g;
        double lb;
        switch (nc) {
        case 2: lb = gmm_em_k<2, KMAX>(x, c, K, n, idx, P, g); break;
        case 3: lb = gmm_em_k<3, KMAX>(x, c, K, n, idx, P, g); break;
        case 4: lb = gmm_em_k<4, KMAX>(x, c, K, n, idx, P, g); break;
        case 5: lb = gmm_em_k<5, KMAX>(x, c, K, n, idx, P, g); break;
        case 6: lb = gmm_em_k<6, KMAX>(x, c, K, n, idx, P, g); break;
        case 7: lb = gmm_em_k<7, KMAX>(x, c, K, n, idx, P, g); break;
        default: lb = gmm_em_k<8, KMAX>(x, c, K, n, idx, P, g); break;
        }
        if (lb > best_lb || best_lb == -INFINITY) best_lb = lb, best = g;
    }
}

// fit_gmm's peak filters (allele.py:88-121) on a fitted nc-component model: the strict weight threshold
// 1 / (filter_factor * nc) always applies for nc > 2; for nc = 2 it is gmm_useless
__device__ __forceinline__ int gmm_useless_k(const GmmK &g, int nc, const AlleleParams &P) {
    double lo = g.mean[0], hi = g.mean[0];
    for (int k = 1; k < nc; ++k) lo = fmin(lo, g.mean[k]), hi = fmax(hi, g.mean[k]);
    const bool strict = nc > 2 || P.force_gm_filter || hi < P.expansion_ratio * fmax(lo, P.small_allele_min);
    const double thr = strict ? 1.0 / (double)(P.filter_factor * nc) : 1.1920928955078125e-07;
    int useless = 0;
    for (int k = 0; k < nc; ++k)
        if (!(g.weight[k] > P.allele_filter && g.weight[k] > thr)) ++useless;
    return useless;
}

// One replicate with A >= 3 alleles (allele.py:56-123,249-293).  fit_gmm's loop: fit with A components, drop the
// useless count and refit with a fresh restart set, a single Gaussian at 1 component, and at <= 0 components the
// last fit with all its components.  A replicate with fewer peaks than A gets A - peaks components drawn with
// probability weight / sum|weight| (Philox stream of the thread), then everything is sorted by mean (stable).
// *n_peaks = the fitted count, before the fill.  forced_init (NULL = k-means++): for nc = A, A-1, ..., 2, n_init
// rows of nc seed indices.  The loop and the bookkeeping are shared with the warp-cooperative fit of deep loci:
// fit(nc, forced, g) is GaussianMixture(nc).fit, single(m, var) make_single_gaussian.
template <class Fit, class Single>
__device__ __forceinline__ void fit_staged(int distinct, int A, const AlleleParams &P, Philox &rng,
                                           const int *forced_init, Fit fit, Single single, double *out_m, double *out_w,
                                           double *out_s, int *n_peaks) {
    GmmK g;
    int nc = distinct == 1 ? 1 : A;  // len(mc) == 1: a single Gaussian without a fit
    while (nc > 1) {
        const int *forced = forced_init ? forced_init + P.n_init * (A * (A + 1) / 2 - nc * (nc + 1) / 2) : nullptr;
        fit(nc, forced, g);
        const int useless = gmm_useless_k(g, nc, P);
        if (!useless) break;
        nc -= useless;
    }
    int peaks;
    if (nc == 1) {
        double m, var;
        single(m, var);
        out_m[0] = m, out_w[0] = 1.0, out_s[0] = sqrt(var);
        peaks = 1;
    } else {
        peaks = g.n_comp;
        for (int k = 0; k < peaks; ++k) out_m[k] = g.mean[k], out_w[k] = g.weight[k], out_s[k] = sqrt(g.cov[k]);
    }
    *n_peaks = peaks;
    if (peaks < A) {
        // Generator.choice(peaks, p = w / sum|w|): cdf normalised by its last entry, searchsorted(side="right")
        double cdf[ALL_MAX_ALLELES], tot = 0.0, acc = 0.0;
        for (int k = 0; k < peaks; ++k) tot += fabs(out_w[k]);
        for (int k = 0; k < peaks; ++k) acc += out_w[k] / tot, cdf[k] = acc;
        for (int k = 0; k < peaks; ++k) cdf[k] /= acc;
        for (int a = peaks; a < A; ++a) {
            int pick = 0;
            if (peaks > 1) {
                const double u = rng.uniform();
                while (pick < peaks - 1 && cdf[pick] <= u) ++pick;
            }
            out_m[a] = out_m[pick], out_w[a] = out_w[pick], out_s[a] = out_s[pick];
        }
    }
    for (int i = 1; i < A; ++i) {  // insertion sort by mean: stable, like argsort(kind="stable")
        const double m = out_m[i], w = out_w[i], s = out_s[i];
        int j = i;
        for (; j > 0 && out_m[j - 1] > m; --j) out_m[j] = out_m[j - 1], out_w[j] = out_w[j - 1], out_s[j] = out_s[j - 1];
        out_m[j] = m, out_w[j] = w, out_s[j] = s;
    }
}

template <int KMAX>
__device__ void fit_replicate_k(const double *x, const int *c, int K, int n, int A, const AlleleParams &P, Philox &rng,
                                const int *forced_init, double *out_m, double *out_w, double *out_s, int *n_peaks) {
    int distinct = 0;
    for (int v = 0; v < K; ++v) distinct += c[v] != 0;
    fit_staged(
        distinct, A, P, rng, forced_init,
        [&](int nc, const int *forced, GmmK &g) { gmm_fit_k<KMAX>(x, c, K, n, nc, P, rng, forced, g); },
        [&](double &m, double &var) { single_gaussian(x, c, K, n, m, var); }, out_m, out_w, out_s, n_peaks);
}

// one replicate of a locus with A alleles: the two-component code for A <= 2, the k-component one above
template <int KMAX, int AMAX>
__device__ __forceinline__ void fit_replicate_any(const double *x, const int *c, int K, int n, int A,
                                                  const AlleleParams &P, Philox &rng, const int *forced_init,
                                                  double *out_m, double *out_w, double *out_s, int *n_peaks) {
    if (AMAX <= 2 || A <= 2)
        fit_replicate<KMAX>(x, c, K, n, A, P, rng, forced_init, out_m, out_w, out_s, n_peaks);
    else
        fit_replicate_k<KMAX>(x, c, K, n, A, P, rng, forced_init, out_m, out_w, out_s, n_peaks);
}

// one thread per (locus, replicate); replicate arrays laid out [locus][allele][replicate] with S allele rows per
// locus; locus l has A_arr[l] alleles (NULL: P.n_alleles).  AMAX = 2 compiles the two-component code only.
template <int KMAX, int AMAX>
__global__ void __launch_bounds__(128)
alleles_fit_kernel(const int *__restrict__ vals, const double *__restrict__ cdf, const int *__restrict__ cnt,
                   const int *__restrict__ K_arr,
                   const int *__restrict__ n_arr, const int *__restrict__ status, const int *__restrict__ A_arr,
                   int n_loci, int kcap, int S, AlleleParams P,
                   double *__restrict__ rep_m, double *__restrict__ rep_w, double *__restrict__ rep_s,
                   unsigned char *__restrict__ rep_peaks) {
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int B = P.num_bootstrap;
    const int l = (int)(tid / B), b = (int)(tid % B);
    if (l >= n_loci || status[l] != 0 || n_arr[l] > ALL_SHALLOW_READS) return;  // deep loci: alleles_deep_fit_kernel
    const int K = K_arr[l], n = n_arr[l];
    if (K > KMAX) return;  // the host picks KMAX >= the batch maximum
    const int A = A_arr ? A_arr[l] : P.n_alleles;
    double x[KMAX];
    int c[KMAX];
    const int *v = vals + (size_t)l * kcap;
    const double *p = cdf + (size_t)l * kcap;
    for (int j = 0; j < K; ++j) x[j] = (double)v[j], c[j] = 0;
    Philox rng;
    rng.init(P.seed, (uint32_t)l, (uint32_t)b);
    if (B > 1) {
        // Generator.choice(replace=True, p): index = cdf.searchsorted(uniform, side="right")
        for (int i = 0; i < n; ++i) {
            const double u = rng.uniform();
            int j = 0;
            while (j < K - 1 && p[j] <= u) ++j;
            ++c[j];
        }
    } else {
        // num_bootstrap == 1: the replicate is the sample itself (allele.py:163-167)
        for (int j = 0; j < K; ++j) c[j] = cnt[(size_t)l * kcap + j];
    }
    double m[AMAX], w[AMAX], s[AMAX];
    int peaks;
    fit_replicate_any<KMAX, AMAX>(x, c, K, n, A, P, rng, nullptr, m, w, s, &peaks);
    for (int a = 0; a < A; ++a) {
        const size_t o = ((size_t)l * S + a) * B + b;
        rep_m[o] = m[a], rep_w[o] = w[a], rep_s[o] = s[a];
    }
    rep_peaks[(size_t)l * B + b] = (unsigned char)peaks;
}

// deterministic building block (tests, and callers that bring their own replicates): problem q has K[q] values
// x[q*kcap ..], counts c[q*kcap ..], and n_init forced seed pairs init[q*2*n_init ..]
template <int KMAX>
__global__ void gmm_fit_counts_kernel(const double *__restrict__ xs, const int *__restrict__ cs, const int *__restrict__ Ks,
                                      const int *__restrict__ init, int n_problems, int kcap, AlleleParams P,
                                      double *__restrict__ out /* [q][7]: m0 w0 s0 m1 w1 s1 peaks */) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n_problems) return;
    const int K = Ks[q];
    if (K > KMAX) return;
    double x[KMAX];
    int c[KMAX], n = 0;
    for (int j = 0; j < K; ++j) x[j] = xs[(size_t)q * kcap + j], c[j] = cs[(size_t)q * kcap + j], n += c[j];
    Philox rng;
    rng.init(P.seed, (uint32_t)q, 0u);
    double m[2] = {0, 0}, w[2] = {0, 0}, s[2] = {0, 0};
    int peaks = 0;
    fit_replicate<KMAX>(x, c, K, n, P.n_alleles, P, rng, init + (size_t)q * 2 * P.n_init, m, w, s, &peaks);
    double *o = out + (size_t)q * 7;
    o[0] = m[0], o[1] = w[0], o[2] = s[0], o[3] = m[1], o[4] = w[1], o[5] = s[1], o[6] = (double)peaks;
}

// the same for problems with their own allele counts A[q] (1..ALL_MAX_ALLELES): seeds init[init_off[q] ..] in
// fit_replicate_k's layout (init = NULL: k-means++ from the problem's Philox stream); out[q][3 * S + 1] =
// means[S], weights[S], stdevs[S] (A[q] of them used, sorted by mean after the fill, the rest 0), n_peaks
template <int KMAX>
__global__ void gmm_fit_counts_ploidy_kernel(const double *__restrict__ xs, const int *__restrict__ cs,
                                             const int *__restrict__ Ks, const int *__restrict__ As,
                                             const int *__restrict__ init, const long long *__restrict__ init_off,
                                             int n_problems, int kcap, int S, AlleleParams P, double *__restrict__ out) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n_problems) return;
    const int K = Ks[q], A = As[q];
    if (K > KMAX) return;
    double x[KMAX];
    int c[KMAX], n = 0;
    for (int j = 0; j < K; ++j) x[j] = xs[(size_t)q * kcap + j], c[j] = cs[(size_t)q * kcap + j], n += c[j];
    Philox rng;
    rng.init(P.seed, (uint32_t)q, 0u);
    double m[ALL_MAX_ALLELES], w[ALL_MAX_ALLELES], s[ALL_MAX_ALLELES];
    int peaks = 0;
    fit_replicate_any<KMAX, ALL_MAX_ALLELES>(x, c, K, n, A, P, rng, init ? init + init_off[q] : nullptr, m, w, s, &peaks);
    double *o = out + (size_t)q * (3 * S + 1);
    for (int a = 0; a < S; ++a) {
        o[a] = a < A ? m[a] : 0.0;
        o[S + a] = a < A ? w[a] : 0.0;
        o[2 * S + a] = a < A ? s[a] : 0.0;
    }
    o[3 * S] = (double)peaks;
}

// ---------------------------------------------------------------------------------------------- deep loci
// Loci with more than ALL_SHALLOW_READS reads.  K can be as large as the read count, so the per-thread arrays above
// do not scale to them: one CTA per deep locus builds its distinct values and CDF in ragged storage, and one warp
// per (locus, replicate) resamples and fits.  A replicate is held as its D nonzero (value, count) pairs in shared
// memory; every sum over them is a lane-strided partial sum followed by a butterfly (xor) reduction, which leaves
// the bitwise same total in every lane, so all lanes carry the same model, the same random state and take the same
// branches.  Given the seeds, the arithmetic per pair is gmm_em_k's; only the order of the sums differs.

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// searchsorted over the cumulative sum of term(0..D): the first j whose inclusive prefix sum is >= r (> r with
// `strict`), D - 1 if none.  32 terms at a time: a shuffle-up scan plus the carry of the chunks before.
template <class T, class Term>
__device__ __forceinline__ int warp_search(int D, T r, bool strict, Term term) {
    const int lane = threadIdx.x & 31;
    T carry = 0;
    for (int j0 = 0; j0 < D; j0 += 32) {
        const int j = j0 + lane;
        T s = j < D ? term(j) : (T)0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const T t = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += t;
        }
        s += carry;
        const unsigned hit = __ballot_sync(0xffffffffu, j < D && (strict ? s > r : s >= r));
        if (hit) return j0 + __ffs(hit) - 1;
        carry = __shfl_sync(0xffffffffu, s, 31);
    }
    return D - 1;
}

// the nonzero counts cnt(0..K) with their values val(j), in ascending j, to cv[0..D) / xv[0..D); returns D.
// cv may be the array cnt reads (every lane reads its entry of a chunk before any lane writes, and writes land at
// or below the chunk).
template <class Cnt, class Val>
__device__ __forceinline__ int warp_compact(int K, Cnt cnt, Val val, double *xv, int *cv) {
    const int lane = threadIdx.x & 31;
    int D = 0;
    for (int j0 = 0; j0 < K; j0 += 32) {
        const int j = j0 + lane;
        const int c = j < K ? cnt(j) : 0;
        const unsigned nz = __ballot_sync(0xffffffffu, c != 0);
        __syncwarp();
        if (c) {
            const int q = D + __popc(nz & ((1u << lane) - 1u));
            cv[q] = c;
            xv[q] = val(j);
        }
        D += __popc(nz);
    }
    __syncwarp();
    return D;
}

// closest squared distance of x to the first nce centres (kmeanspp_k's running fmin, recomputed)
__device__ __forceinline__ double closest_sq(double x, const double *cen, int nce) {
    double d = x - cen[0], cl = d * d;
#pragma unroll
    for (int i = 1; i < ALL_MAX_ALLELES; ++i)
        if (i < nce) d = x - cen[i], cl = fmin(cl, d * d);
    return cl;
}

// kmeanspp_k on D nonzero pairs, warp-cooperative: the centres' values to cen[0..k)
__device__ void kmeanspp_warp(const double *xv, const int *cv, int D, int n, int k, Philox &rng, double *cen) {
    const int lane = threadIdx.x & 31;
    {
        const double u = rng.uniform();
        long long pt = (long long)(u * (double)n);
        if (pt >= n) pt = n - 1;
        cen[0] = xv[warp_search<long long>(D, pt, true, [&](int j) { return (long long)cv[j]; })];
    }
    double pot = 0.0;
    for (int j = lane; j < D; j += 32) pot += (double)cv[j] * closest_sq(xv[j], cen, 1);
    pot = warp_sum(pot);
    const int trials = 2 + (int)log((double)k);
    for (int ci = 1; ci < k; ++ci) {
        double best_pot = INFINITY;
        int best = 0;
#pragma unroll 1
        for (int t = 0; t < trials; ++t) {
            const double r = rng.uniform() * pot;
            const int cand = warp_search<double>(D, r, false,
                                                 [&](int j) { return (double)cv[j] * closest_sq(xv[j], cen, ci); });
            double cp = 0.0;
            for (int j = lane; j < D; j += 32) {
                const double d = xv[j] - xv[cand];
                cp += (double)cv[j] * fmin(closest_sq(xv[j], cen, ci), d * d);
            }
            cp = warp_sum(cp);
            if (cp < best_pot) best_pot = cp, best = cand;
        }
        cen[ci] = xv[best];
        pot = best_pot;
    }
}

// gmm_em_k from the seed values cen[0..NC) on D nonzero pairs, warp-cooperative
template <int NC>
__device__ double gmm_em_warp(const double *xv, const int *cv, int D, int n, const double *cen, const AlleleParams &P,
                              GmmK &g) {
    const int lane = threadIdx.x & 31;
    const double eps10 = 10.0 * 2.220446049250313e-16;
    double mean[NC], cov[NC], weight[NC], pchol[NC], logw[NC];
#pragma unroll
    for (int k = 0; k < NC; ++k) {
        const double nk = 1.0 + eps10, xk = cen[k];
        mean[k] = xk / nk;
        cov[k] = __dadd_rn(__dsub_rn(__ddiv_rn(__dmul_rn(xk, xk), nk), __dmul_rn(mean[k], mean[k])), P.reg_covar);
        weight[k] = nk / (double)n;
        pchol[k] = 1.0 / sqrt(cov[k]);
        logw[k] = log(weight[k]);
    }
    double lower = -INFINITY;
    for (int it = 1; it <= P.max_iter; ++it) {
        const double prev = lower;
        double nk[NC], sx[NC], sxx[NC], ll = 0.0;
#pragma unroll
        for (int k = 0; k < NC; ++k) nk[k] = 0.0, sx[k] = 0.0, sxx[k] = 0.0;
        for (int j = lane; j < D; j += 32) {
            const double x = xv[j];
            double wl[NC];
#pragma unroll
            for (int k = 0; k < NC; ++k) wl[k] = gmm_wlp1(x, mean[k], pchol[k], logw[k]);
            double mx = wl[0];
#pragma unroll
            for (int k = 1; k < NC; ++k) mx = fmax(mx, wl[k]);
            double se = 0.0;
#pragma unroll
            for (int k = 0; k < NC; ++k) se += exp(wl[k] - mx);
            const double lse = mx + log(se);
            const double c = (double)cv[j];
            ll += c * lse;
#pragma unroll
            for (int k = 0; k < NC; ++k) {
                const double r = exp(wl[k] - lse) * c;
                nk[k] += r;
                sx[k] += r * x;
                sxx[k] += r * x * x;
            }
        }
        ll = warp_sum(ll);
#pragma unroll
        for (int k = 0; k < NC; ++k) nk[k] = warp_sum(nk[k]), sx[k] = warp_sum(sx[k]), sxx[k] = warp_sum(sxx[k]);
        lower = ll / (double)n;
        double wsum = 0.0;
#pragma unroll
        for (int k = 0; k < NC; ++k) {
            nk[k] += eps10;
            mean[k] = sx[k] / nk[k];
            cov[k] = __dadd_rn(__dsub_rn(__ddiv_rn(sxx[k], nk[k]), __dmul_rn(mean[k], mean[k])), P.reg_covar);
            weight[k] = nk[k] / (double)n;
            wsum += weight[k];
        }
#pragma unroll
        for (int k = 0; k < NC; ++k) {
            weight[k] /= wsum;
            pchol[k] = 1.0 / sqrt(cov[k] > 0.0 ? cov[k] : P.reg_covar);
            logw[k] = log(weight[k]);
        }
        if (fabs(lower - prev) < P.tol) break;
    }
#pragma unroll
    for (int k = 0; k < NC; ++k) g.mean[k] = mean[k], g.cov[k] = cov[k], g.weight[k] = weight[k];
    g.n_comp = NC;
    return lower;
}

// gmm_fit_k, warp-cooperative: forced seed indices point into x_forced (the caller's value list)
__device__ void gmm_fit_warp(const double *xv, const int *cv, int D, int n, int nc, const AlleleParams &P, Philox &rng,
                             const int *forced, const double *x_forced, GmmK &best) {
    double best_lb = -INFINITY;
    for (int t = 0; t < P.n_init; ++t) {
        double cen[ALL_MAX_ALLELES];
        if (forced) {
            for (int j = 0; j < nc; ++j) cen[j] = x_forced[forced[t * nc + j]];
        } else {
            kmeanspp_warp(xv, cv, D, n, nc, rng, cen);
        }
        GmmK g;
        double lb;
        switch (nc) {
        case 2: lb = gmm_em_warp<2>(xv, cv, D, n, cen, P, g); break;
        case 3: lb = gmm_em_warp<3>(xv, cv, D, n, cen, P, g); break;
        case 4: lb = gmm_em_warp<4>(xv, cv, D, n, cen, P, g); break;
        case 5: lb = gmm_em_warp<5>(xv, cv, D, n, cen, P, g); break;
        case 6: lb = gmm_em_warp<6>(xv, cv, D, n, cen, P, g); break;
        case 7: lb = gmm_em_warp<7>(xv, cv, D, n, cen, P, g); break;
        default: lb = gmm_em_warp<8>(xv, cv, D, n, cen, P, g); break;
        }
        if (lb > best_lb || best_lb == -INFINITY) best_lb = lb, best = g;
    }
}

// One replicate of a deep locus (any A, 1..8): fit_gmm's staged loop and bookkeeping (fit_staged) over the warp
// fits.  For A <= 2 this is the two-component code's result too: the staged loop at 2 components is fit_replicate
// (the same k-means++ draws, EM and filter).
__device__ void fit_replicate_warp(const double *xv, const int *cv, int D, int n, int A, const AlleleParams &P,
                                   Philox &rng, const int *forced_init, const double *x_forced, double *out_m,
                                   double *out_w, double *out_s, int *n_peaks) {
    const int lane = threadIdx.x & 31;
    fit_staged(
        D, A, P, rng, forced_init,
        [&](int nc, const int *forced, GmmK &g) { gmm_fit_warp(xv, cv, D, n, nc, P, rng, forced, x_forced, g); },
        [&](double &m, double &var) {
            double s = 0.0;
            for (int j = lane; j < D; j += 32) s += (double)cv[j] * xv[j];
            m = warp_sum(s) / (double)n;
            double q = 0.0;
            for (int j = lane; j < D; j += 32) {
                const double d = xv[j] - m;
                q += (double)cv[j] * d * d;
            }
            var = warp_sum(q) / (double)n;
        },
        out_m, out_w, out_s, n_peaks);
}

// one CTA per deep locus deep_l[d]: its sorted distinct values and resampling CDF at deep_off[d] (ragged, up to
// ALL_DEEP_MAX_K entries), K, status (1: fewer than min_reads reads, 2: one distinct value, else 0; fewer reads
// than A cannot occur above ALL_SHALLOW_READS reads), and its first value at vals[l * kcap], where the aggregation
// reads the value of a status-2 locus.  More than ALL_DEEP_MAX_K distinct values: deep_K[d] > ALL_DEEP_MAX_K and
// nothing else is written (the host reports the locus).
// The per-value weight sums are fixed-point integers (each weight scaled to 2^63 / (n * max weight) and rounded):
// integer atomics make them independent of the order the threads add in, and the CDF of exact integer sums is
// cdf[j] = sum[0..j] / sum[0..K), normalised by the total as Generator.choice does (cdf /= cdf[-1]).
#define ALL_DEEP_TABLE (2 * ALL_DEEP_MAX_K)  // open-addressing hash set of the distinct values (load <= 0.53)
__global__ void __launch_bounds__(256)
alleles_deep_prepare_kernel(const int *__restrict__ cn, const double *__restrict__ w,
                            const long long *__restrict__ read_begin, const int *__restrict__ deep_l,
                            const long long *__restrict__ deep_off, int min_reads, int kcap, int *__restrict__ dvals,
                            double *__restrict__ dcdf, int *__restrict__ K_out, int *__restrict__ deep_K,
                            int *__restrict__ status, int *__restrict__ vals) {
    extern __shared__ unsigned long long smem_deep_prep[];
    unsigned long long *table = smem_deep_prep;                  // [ALL_DEEP_TABLE]; then wsum[ALL_DEEP_MAX_K]
    int *sv = (int *)(smem_deep_prep + ALL_DEEP_TABLE);          // [ALL_DEEP_MAX_K] sorted distinct values
    __shared__ int s_K, s_slot;
    __shared__ double s_wmax;
    const unsigned long long EMPTY = ~0ull;
    const int d = blockIdx.x, l = deep_l[d];
    const long long r0 = read_begin[l], r1 = read_begin[l + 1];
    const int n = (int)(r1 - r0);
    for (int i = threadIdx.x; i < ALL_DEEP_TABLE; i += blockDim.x) table[i] = EMPTY;
    if (threadIdx.x == 0) s_K = 0, s_slot = 0, s_wmax = 0.0;
    __syncthreads();
    // distinct values; a thread stops once the set is over the cap, so at most cap + blockDim entries are inserted
    double wmax = 0.0;
    for (long long r = r0 + threadIdx.x; r < r1; r += blockDim.x) {
        wmax = fmax(wmax, w[r]);
        if (*(volatile int *)&s_K > ALL_DEEP_MAX_K) continue;
        const unsigned long long key = (unsigned)cn[r];
        unsigned h = ((unsigned)cn[r] * 2654435761u) & (ALL_DEEP_TABLE - 1);
        for (;;) {
            const unsigned long long old = atomicCAS(&table[h], EMPTY, key);
            if (old == EMPTY) {
                atomicAdd(&s_K, 1);
                break;
            }
            if (old == key) break;
            h = (h + 1) & (ALL_DEEP_TABLE - 1);
        }
    }
    // weights are >= 0: their doubles order like their bit patterns
    atomicMax((unsigned long long *)&s_wmax, (unsigned long long)__double_as_longlong(wmax));
    __syncthreads();
    const int K = s_K;
    if (K > ALL_DEEP_MAX_K) {
        if (threadIdx.x == 0) deep_K[d] = K;
        return;
    }
    int np2 = 1;
    while (np2 < K) np2 <<= 1;
    for (int i = threadIdx.x; i < ALL_DEEP_TABLE; i += blockDim.x)
        if (table[i] != EMPTY) sv[atomicAdd(&s_slot, 1)] = (int)(unsigned)table[i];
    for (int i = K + threadIdx.x; i < np2; i += blockDim.x) sv[i] = 0x7fffffff;
    __syncthreads();
    for (int k = 2; k <= np2; k <<= 1)  // bitonic sort of the distinct values (slot order above is arbitrary)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = threadIdx.x; t < np2; t += blockDim.x) {
                const int u = t ^ j;
                if (u > t) {
                    const int a = sv[t], b = sv[u];
                    if ((a > b) == ((t & k) == 0)) sv[t] = b, sv[u] = a;
                }
            }
            __syncthreads();
        }
    unsigned long long *wsum = table;
    for (int j = threadIdx.x; j < K; j += blockDim.x) wsum[j] = 0;
    __syncthreads();
    const double scale = s_wmax > 0.0 ? 9223372036854775808.0 / ((double)n * s_wmax) : 0.0;
    for (long long r = r0 + threadIdx.x; r < r1; r += blockDim.x) {
        const int x = cn[r];
        int lo = 0, hi = K - 1;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (sv[mid] < x) lo = mid + 1;
            else hi = mid;
        }
        const double wr = w[r];
        atomicAdd(&wsum[lo], (unsigned long long)rint((wr > 0.0 ? wr : 0.0) * scale));
    }
    __syncthreads();
    if (threadIdx.x == 0)
        for (int j = 1; j < K; ++j) wsum[j] += wsum[j - 1];
    __syncthreads();
    const double tot = (double)wsum[K - 1];
    int *v = dvals + deep_off[d];
    double *p = dcdf + deep_off[d];
    for (int j = threadIdx.x; j < K; j += blockDim.x) v[j] = sv[j], p[j] = (double)wsum[j] / tot;
    if (threadIdx.x == 0) {
        deep_K[d] = K_out[l] = K;
        status[l] = n < min_reads ? 1 : (K == 1 ? 2 : 0);
        vals[(size_t)l * kcap] = sv[0];
    }
}

// one warp per (deep locus, replicate): CTA (d, y) takes replicates y * ALL_DEEP_WARPS + warp of deep locus deep_l[d].
// Shared memory: the locus' CDF [K], then per warp the replicate's counts [K] (int) and its compacted values [K].
// Resampling: draw i of replicate b is uniform i of the Philox stream (seed, l, b | ALL_DEEP_STREAM) from counter
// (0, 0), two per counter, and searchsorted(cdf, u, side="right") by binary search; the lanes take alternate
// counters and add to the warp's counts with integer atomics.  The fit draws from the same key from counter (0, 1).
// Keys are the batch's seed and locus index, not the chunk's, so a deep row depends on neither the chunking nor the
// launch shape.  Rows go to the chunk's replicate scratch at locus l - l0.
__global__ void __launch_bounds__(32 * ALL_DEEP_WARPS)
alleles_deep_fit_kernel(const int *__restrict__ deep_l, const long long *__restrict__ deep_off,
                        const int *__restrict__ dvals, const double *__restrict__ dcdf, const int *__restrict__ K_arr,
                        const int *__restrict__ n_arr, const int *__restrict__ status, const int *__restrict__ A_arr,
                        int l0, int S, AlleleParams P, double *__restrict__ rep_m, double *__restrict__ rep_w,
                        double *__restrict__ rep_s, unsigned char *__restrict__ rep_peaks) {
    extern __shared__ double smem_deep_fit[];
    const int d = blockIdx.x, l = deep_l[d];
    if (status[l] != 0) return;
    const int K = K_arr[l], n = n_arr[l], B = P.num_bootstrap;
    const int A = A_arr ? A_arr[l] : P.n_alleles;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double *cdf = smem_deep_fit;
    double *xv = cdf + (size_t)K * (1 + warp);
    int *cv = (int *)(cdf + (size_t)K * (1 + ALL_DEEP_WARPS)) + (size_t)K * warp;
    const int *v = dvals + deep_off[d];
    const double *p = dcdf + deep_off[d];
    for (int j = threadIdx.x; j < K; j += blockDim.x) cdf[j] = p[j];
    for (int j = lane; j < K; j += 32) cv[j] = 0;
    __syncthreads();
    const int b = blockIdx.y * ALL_DEEP_WARPS + warp;
    if (b >= B) return;
    Philox rng;
    rng.init(P.seed, (uint32_t)l, (uint32_t)b | ALL_DEEP_STREAM);
    for (unsigned pr = lane; pr < ((unsigned)n + 1u) / 2u; pr += 32) {
        rng.seek(pr, 0u);
        for (int h = 0; h < 2 && 2 * (long long)pr + h < n; ++h) {
            const double u = rng.uniform();
            int lo = 0, hi = K - 1;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (cdf[mid] <= u) lo = mid + 1;
                else hi = mid;
            }
            atomicAdd(&cv[lo], 1);
        }
    }
    __syncwarp();
    const int D = warp_compact(K, [&](int j) { return cv[j]; }, [&](int j) { return (double)v[j]; }, xv, cv);
    rng.seek(0u, 1u);
    double m[ALL_MAX_ALLELES], w[ALL_MAX_ALLELES], s[ALL_MAX_ALLELES];
    int peaks;
    fit_replicate_warp(xv, cv, D, n, A, P, rng, nullptr, nullptr, m, w, s, &peaks);
    if (lane == 0) {
        const size_t ll = (size_t)(l - l0);
        for (int a = 0; a < A; ++a) {
            const size_t o = (ll * S + a) * B + b;
            rep_m[o] = m[a], rep_w[o] = w[a], rep_s[o] = s[a];
        }
        rep_peaks[ll * B + b] = (unsigned char)peaks;
    }
}

// gmm_fit_counts_ploidy_kernel through the warp fit, for any K up to kcap <= ALL_DEEP_MAX_K: one warp per problem,
// its nonzero (value, count) pairs in shared memory ([warp][kcap] values, then [warp][kcap] counts); the stream of
// problem q is (seed, q, ALL_DEEP_STREAM) from counter (0, 1), as a deep replicate's fit
__global__ void __launch_bounds__(32 * ALL_DEEP_WARPS)
gmm_fit_counts_deep_kernel(const double *__restrict__ xs, const int *__restrict__ cs, const int *__restrict__ Ks,
                           const int *__restrict__ As, const int *__restrict__ init,
                           const long long *__restrict__ init_off, int n_problems, int kcap, int S, AlleleParams P,
                           double *__restrict__ out) {
    extern __shared__ double smem_deep_fit[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = blockIdx.x * ALL_DEEP_WARPS + warp;
    if (q >= n_problems) return;
    double *xv = smem_deep_fit + (size_t)kcap * warp;
    int *cv = (int *)(smem_deep_fit + (size_t)kcap * ALL_DEEP_WARPS) + (size_t)kcap * warp;
    const double *x = xs + (size_t)q * kcap;
    const int *c = cs + (size_t)q * kcap;
    const int D = warp_compact(Ks[q], [&](int j) { return c[j]; }, [&](int j) { return x[j]; }, xv, cv);
    int n = 0;
    for (int j = lane; j < D; j += 32) n += cv[j];
    n = __reduce_add_sync(0xffffffffu, n);
    Philox rng;
    rng.init(P.seed, (uint32_t)q, ALL_DEEP_STREAM);
    rng.seek(0u, 1u);
    double m[ALL_MAX_ALLELES], w[ALL_MAX_ALLELES], s[ALL_MAX_ALLELES];
    int peaks = 0;
    const int A = As[q];
    fit_replicate_warp(xv, cv, D, n, A, P, rng, init ? init + init_off[q] : nullptr, x, m, w, s, &peaks);
    if (lane == 0) {
        double *o = out + (size_t)q * (3 * S + 1);
        for (int a = 0; a < S; ++a) {
            o[a] = a < A ? m[a] : 0.0;
            o[S + a] = a < A ? w[a] : 0.0;
            o[2 * S + a] = a < A ? s[a] : 0.0;
        }
        o[3 * S] = (double)peaks;
    }
}

// ---------------------------------------------------------------------------------------------- aggregate
// np.percentile(..., method="interpolated_inverted_cdf") on an ascending array a[0..n): virtual index n*q - 1
__device__ __forceinline__ double pct_iicdf(const double *a, int n, double q) {
    double vi = (double)n * q - 1.0;
    if (vi < 0.0) vi = 0.0;
    if (vi > (double)(n - 1)) vi = (double)(n - 1);
    const int lo = (int)floor(vi);
    const int hi = lo + 1 < n ? lo + 1 : n - 1;
    const double g = vi - (double)lo;
    // numpy _lerp: a + (b - a) * t, switched to b - (b - a) * (1 - t) for t >= 0.5
    const double d = a[hi] - a[lo];
    return g >= 0.5 ? a[hi] - d * (1.0 - g) : a[lo] + d * g;
}

// out_i [locus][1 + 2*S + 4*S]: modal_n, call[S], ci95[S][2], ci99[S][2]      out_d [locus][3*S]: means, weights,
// stdevs.  Locus l has A = A_arr[l] alleles (NULL: S) in replicate rows [locus][S][B]; its columns A..S-1 are 0.
__global__ void __launch_bounds__(256)
alleles_aggregate_kernel(const double *__restrict__ rep_m, const double *__restrict__ rep_w, const double *__restrict__ rep_s,
                         const unsigned char *__restrict__ rep_peaks, const int *__restrict__ status,
                         const int *__restrict__ vals, int kcap, int n_loci, const int *__restrict__ A_arr, int S, int B,
                         int *__restrict__ out_i, double *__restrict__ out_d) {
    extern __shared__ unsigned char smem_raw_all[];
    const int l = blockIdx.x;
    if (l >= n_loci) return;
    int np2 = 1;
    while (np2 < B) np2 <<= 1;
    double *key = (double *)smem_raw_all;  // [np2] replicate means of one allele
    int *idx = (int *)(key + np2);         // [np2] replicate index (tie-break = stable order)
    int *oi = out_i + (size_t)l * (1 + 5 * S);
    double *od = out_d + (size_t)l * (3 * S);
    const int A = A_arr ? A_arr[l] : S;
    for (int a = A + threadIdx.x; a < S; a += blockDim.x) {
        oi[1 + a] = 0;
        oi[1 + S + 2 * a] = oi[1 + S + 2 * a + 1] = 0;
        oi[1 + 3 * S + 2 * a] = oi[1 + 3 * S + 2 * a + 1] = 0;
        od[a] = od[S + a] = od[2 * S + a] = 0.0;
    }
    const int st = status[l];
    if (st != 0) {
        if (threadIdx.x == 0) {
            const int cnv = st == 2 ? vals[(size_t)l * kcap] : 0;
            oi[0] = st == 2 ? 1 : 0;
            for (int a = 0; a < A; ++a) {
                oi[1 + a] = cnv;
                oi[1 + S + 2 * a] = oi[1 + S + 2 * a + 1] = cnv;
                oi[1 + 3 * S + 2 * a] = oi[1 + 3 * S + 2 * a + 1] = cnv;
                od[a] = (double)cnv;
                od[S + a] = st == 2 ? 1.0 / (double)A : 0.0;
                od[2 * S + a] = 0.0;
            }
        }
        return;
    }
    __shared__ int s_cnt[256];  // replicates per peak count
    s_cnt[threadIdx.x] = 0;
    __syncthreads();
    for (int b = threadIdx.x; b < B; b += blockDim.x) atomicAdd(&s_cnt[rep_peaks[(size_t)l * B + b]], 1);
    __syncthreads();
    double wsel[ALL_MAX_ALLELES];
    for (int a = 0; a < A; ++a) {
        const double *m = rep_m + ((size_t)l * S + a) * B;
        for (int b = threadIdx.x; b < np2; b += blockDim.x) {
            key[b] = b < B ? m[b] : INFINITY;
            idx[b] = b;
        }
        __syncthreads();
        // bitonic sort of (key, original index): lexicographic order = numpy's stable argsort
        for (int k = 2; k <= np2; k <<= 1)
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int t = threadIdx.x; t < np2; t += blockDim.x) {
                    const int u = t ^ j;
                    if (u > t) {
                        const bool up = (t & k) == 0;
                        const double ka = key[t], kb = key[u];
                        const int ia = idx[t], ib = idx[u];
                        const bool gt = ka > kb || (ka == kb && ia > ib);
                        if (gt == up) key[t] = kb, key[u] = ka, idx[t] = ib, idx[u] = ia;
                    }
                }
                __syncthreads();
            }
        if (threadIdx.x == 0) {
            const int med = B / 2;
            const size_t o = ((size_t)l * S + a) * B + idx[med];
            od[a] = key[med];
            wsel[a] = rep_w[o];
            od[2 * S + a] = rep_s[o];
            oi[1 + a] = (int)rint(key[med]);
            oi[1 + S + 2 * a] = (int)rint(pct_iicdf(key, B, 0.025));
            oi[1 + S + 2 * a + 1] = (int)rint(pct_iicdf(key, B, 0.975));
            oi[1 + 3 * S + 2 * a] = (int)rint(pct_iicdf(key, B, 0.005));
            oi[1 + 3 * S + 2 * a + 1] = (int)rint(pct_iicdf(key, B, 0.995));
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        double ws = 0.0;
        for (int a = 0; a < A; ++a) ws += wsel[a];
        for (int a = 0; a < A; ++a) od[S + a] = wsel[a] / ws;
        // statistics.mode of the sorted peak counts: the smallest of the most common
        int modal = 0;
        for (int k = 1; k < 256; ++k)
            if (s_cnt[k] > s_cnt[modal]) modal = k;
        oi[0] = modal;
    }
}
