// realign_api.cuh -- C ABI of the soft-clip realignment (included at the end of api.cu).
#pragma once
#include "realign.cuh"

extern "C" int strk_realign(strk_ctx *ctx, const uint8_t *arena, uint64_t arena_bytes, const uint64_t *ref_off,
                            const int32_t *ref_len, const uint64_t *read_off, const int32_t *read_len, int64_t n,
                            int gap_open, int gap_extend, int trace_flags, int32_t *score, int32_t *end_ref,
                            uint32_t *cigar, const uint64_t *cigar_off, int32_t *cigar_len) {
    if (!ctx || !arena || !ref_off || !ref_len || !read_off || !read_len || !score || !end_ref || !cigar || !cigar_off ||
        !cigar_len)
        return set_err(STRK_ERR_ARG, "strk_realign: null argument");
    if (n <= 0 || n > (1 << 24)) return set_err(STRK_ERR_ARG, "strk_realign: bad alignment count");
    if (gap_open < 0 || gap_extend < 0 || gap_open > 1000 || gap_extend > 1000)
        return set_err(STRK_ERR_ARG, "strk_realign: bad gap penalties");
    std::vector<RealignDesc> descs((size_t)n);
    int max_n2 = 0;
    for (int64_t k = 0; k < n; ++k) {
        const int n1 = ref_len[k], n2 = read_len[k];
        if (n1 <= 0 || n2 <= 0 || n1 > (1 << 20) || n2 > (1 << 24))
            return set_err(STRK_ERR_ARG, "strk_realign: alignment %lld has an empty or oversized sequence", (long long)k);
        if (ref_off[k] + (uint64_t)n1 > arena_bytes || read_off[k] + (uint64_t)n2 > arena_bytes)
            return set_err(STRK_ERR_ARG, "strk_realign: alignment %lld runs past the end of the arena", (long long)k);
        if ((int64_t)(cigar_off[k + 1] - cigar_off[k]) < 2 * (int64_t)n1 + 4)
            return set_err(STRK_ERR_ARG, "strk_realign: cigar region of alignment %lld is smaller than 2 * len(ref) + 4",
                           (long long)k);
        RealignDesc &d = descs[(size_t)k];
        d.s1_off = ref_off[k], d.s2_off = read_off[k], d.n1 = n1, d.n2 = n2;
        d.cigar_off = cigar_off[k];
        d.cigar_cap = (int)std::min<uint64_t>(cigar_off[k + 1] - cigar_off[k], 0x7fffffffu);
        d.R = ra_pick_rows(n1);
        d.NB = (n1 + 32 * d.R - 1) / (32 * d.R);
        max_n2 = std::max(max_n2, n2);
    }
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    // groups of alignments whose traces fit the budget (1 byte per cell; STRK_REALIGN_TRACE_MB, default 2048)
    size_t budget = 2048ull << 20;
    if (const char *e = getenv("STRK_REALIGN_TRACE_MB")) budget = (size_t)std::max(1, atoi(e)) << 20;
    TmpDev tmp{st};
    unsigned char *d_arena = nullptr;
    cudaError_t e = tmp.up(&d_arena, arena, (size_t)arena_bytes);
    const uint64_t cigar_total = cigar_off[n];
    unsigned int *d_cigar = nullptr;
    int *d_score = nullptr, *d_end = nullptr, *d_len = nullptr;
    RealignDesc *d_descs = nullptr;
    unsigned int *d_q = nullptr;
    if (e == cudaSuccess) e = tmp.get(&d_cigar, (size_t)cigar_total);
    if (e == cudaSuccess) e = tmp.get(&d_score, (size_t)n);
    if (e == cudaSuccess) e = tmp.get(&d_end, (size_t)n);
    if (e == cudaSuccess) e = tmp.get(&d_len, (size_t)n);
    if (e == cudaSuccess) e = tmp.get(&d_descs, (size_t)n);
    if (e == cudaSuccess) e = tmp.get(&d_q, 1);
    const int grid_max = ctx->n_sm * 4;
    const int bound_stride = 4 * (max_n2 + 1);
    int *d_bound = nullptr;
    if (e == cudaSuccess) e = tmp.get(&d_bound, (size_t)grid_max * RA_WARPS * (size_t)bound_stride);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(STRK_ERR_NOMEM, "strk_realign: %s", cudaGetErrorString(e));
    }
    unsigned char *d_trace = nullptr;
    size_t trace_cap = 0;
    for (int k = 0; k < 8; ++k) ctx->stats[k] = 0;
    double cells = 0.0;
    float ms_total = 0.f;
    int64_t k0 = 0;
    while (k0 < n) {
        size_t used = 0;
        int64_t k1 = k0;
        while (k1 < n) {
            const size_t need = (size_t)ra_trace_bytes(descs[(size_t)k1].n1, descs[(size_t)k1].n2);
            if (k1 > k0 && used + need > budget) break;
            descs[(size_t)k1].trace_off = used;
            used += (need + 15) / 16 * 16;
            cells += (double)descs[(size_t)k1].n1 * (double)descs[(size_t)k1].n2;
            ++k1;
        }
        if (used > trace_cap) {
            if (d_trace) cudaFree(d_trace);
            d_trace = nullptr;
            if (cudaMalloc((void **)&d_trace, used) != cudaSuccess) {
                cudaGetLastError();
                return set_err(STRK_ERR_NOMEM, "strk_realign: cannot allocate %zu bytes of traceback (1 byte per DP cell; "
                                               "lower STRK_REALIGN_TRACE_MB or split the call)", used);
            }
            trace_cap = used;
        }
        const int cnt = (int)(k1 - k0);
        int rc = STRK_OK;
        auto fail = [&](cudaError_t ce, const char *what) {
            rc = set_err(STRK_ERR_CUDA, "strk_realign: %s: %s", what, cudaGetErrorString(ce));
        };
        cudaError_t ce = cudaMemcpyAsync(d_descs + k0, descs.data() + k0, (size_t)cnt * sizeof(RealignDesc),
                                         cudaMemcpyHostToDevice, st);
        if (ce == cudaSuccess) ce = cudaMemsetAsync(d_q, 0, sizeof(unsigned int), st);
        if (ce == cudaSuccess) ce = cudaEventRecord(ctx->ev[0], st);
        if (ce == cudaSuccess) {
            const int grid = std::min(grid_max, (cnt + RA_WARPS - 1) / RA_WARPS);
            realign_fill_kernel<<<grid, RA_WARPS * 32, 0, st>>>(d_descs + k0, cnt, d_arena, ctx->d_consts, d_trace, d_bound,
                                                                bound_stride, gap_open, gap_extend, trace_flags,
                                                                d_score + k0, d_end + k0, d_q);
            ce = cudaGetLastError();
        }
        if (ce == cudaSuccess) {
            realign_trace_kernel<<<(cnt + 63) / 64, 64, 0, st>>>(d_descs + k0, cnt, d_arena, ctx->d_consts, d_trace,
                                                                 d_end + k0, d_cigar, d_len + k0);
            ce = cudaGetLastError();
        }
        if (ce == cudaSuccess) ce = cudaEventRecord(ctx->ev[1], st);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
        if (ce != cudaSuccess) fail(ce, "kernels");
        if (rc) {
            if (d_trace) cudaFree(d_trace);
            return rc;
        }
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
        ms_total += ms;
        ctx->stats[2] += 2;
        k0 = k1;
    }
    if (d_trace) cudaFree(d_trace);
    CU(cudaMemcpy(score, d_score, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(end_ref, d_end, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(cigar_len, d_len, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(cigar, d_cigar, (size_t)cigar_total * sizeof(unsigned int), cudaMemcpyDeviceToHost));
    for (int64_t k = 0; k < n; ++k) {
        end_ref[k] -= 1;  // parasail end_ref: 0-based last read position aligned (-1: the window met no read base)
        if (cigar_len[k] < 0) return set_err(STRK_ERR_ARG, "strk_realign: cigar region of alignment %lld overflowed", (long long)k);
    }
    ctx->stats[0] = cells;
    ctx->stats[3] = ms_total;
    return STRK_OK;
}
