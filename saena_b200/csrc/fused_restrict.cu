// fused_restrict.cu -- MEASUREMENT of the north_star's "restriction fused with the residual that feeds it".
//
// Reference: the V-cycle computes res = A u - rhs (src/saena_object_solve.cpp:1140, saena_matrix::residual,
// include/saena_matrix.tpp:16-23) and then res_coarse = R res (:1175, restrict_matrix::matvec_sparse,
// src/restrict_matrix.cpp:612-744), R = P^T entry for entry (restrict_matrix::transposeP, :229-494).
//
// Fusing the two means never writing `res`: the thread that finishes (A u - rhs)_i scatters it through row i of P,
// res_coarse[c] += P[i,c] * res_i, with FP64 atomics (the gather form would recompute every fine residual once per
// coarse row that touches it, ~6x the A traffic).  It saves the write and the re-read of res (16 B per fine row) and
// costs nnz(P) atomic adds plus a zero-fill of res_coarse.  The solve path keeps the two kernels; this file exists so
// that the decision rests on a measurement (profiles/r02_fused_restrict.md), not on an estimate: it times both forms
// on an uploaded level and compares their results.  One rank, A on the sliced layout (levels 0-2 of the bench
// hierarchy: the levels whose res does not stay in L2), P with 32-bit row offsets.
#include <algorithm>
#include <vector>

#include "spmv_kernels.cuh"

__global__ void __launch_bounds__(256)
residual_restrict_sell_kernel(int M, const long long *__restrict__ slice_ptr, const int *__restrict__ col,
                              const double *__restrict__ val, const double *__restrict__ x,
                              const double *__restrict__ rhs, const int *__restrict__ p_rowptr,
                              const int *__restrict__ p_col, const double *__restrict__ p_val,
                              double *__restrict__ res_coarse) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const int slice = row >> 5;
    if ((slice << 5) >= M) return;
    const long long base = slice_ptr[slice];
    const int len = (int)((slice_ptr[slice + 1] - base) >> 5);
    const int *cp = col + base + lane;
    const double *vp = val + base + lane;
    double sum = 0.0;
    int j = 0;
    for (; j + 4 <= len; j += 4) {
        int c[4];
        double a[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            c[q] = sb_ld_stream(cp + (j + q) * 32);
            a[q] = sb_ld_stream(vp + (j + q) * 32);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) sum += a[q] * __ldg(x + c[q]);
    }
    for (; j < len; ++j) sum += sb_ld_stream(vp + j * 32) * __ldg(x + sb_ld_stream(cp + j * 32));
    if (row >= M) return;
    const double r = sum - rhs[row];                       // saena_matrix.tpp:16-23
    const int a = p_rowptr[row], b = p_rowptr[row + 1];    // row i of P = column i of R
    for (int k = a; k < b; ++k) atomicAdd(res_coarse + p_col[k], p_val[k] * r);
}

// The fused form inside the V-cycle (opt-in, saena_b200_set_fused_restrict): res_coarse = R (A u - rhs) in one pass over
// A, `res` never written.  Eligible: no halo on A, P, R of the level (one rank, or an agglomerated level), A on the
// sliced layout, P with 32-bit CSR arrays.  Returns 1 when it ran, 0 when the level is not eligible (the caller runs
// the two kernels), < 0 on error.
int sb_residual_restrict_fused(saena_b200_ctx *ctx, int l, const double *u, const double *rhs, double *res_coarse) {
    DevLevel &lv = ctx->levels[l];
    DevOperator &A = lv.A, &P = lv.P, &R = lv.R;
    if (l >= ctx->fused_restrict_levels) return 0;
    if (A.mapping != SB_MAPPING_SELL || !A.sell.ptr || !P.present || P.wide_offsets || !P.col || !P.val || P.merged || R.merged) return 0;
    if (!A.sends.empty() || !A.recvs.empty() || !P.sends.empty() || !P.recvs.empty() || !R.sends.empty() || !R.recvs.empty()) return 0;
    if (A.nnz_remote || P.nnz_remote || R.nnz_remote || lv.M == 0) return 0;
    if (cudaMemsetAsync(res_coarse, 0, sizeof(double) * (size_t)std::max(R.M, 1), ctx->stream) != cudaSuccess) return -1;
    ctx->launches += 1;
    residual_restrict_sell_kernel<<<(lv.M + 255) / 256, 256, 0, ctx->stream>>>(lv.M, A.sell.ptr, A.sell.col, A.sell.val, u, rhs,
                                                                          (const int *)P.rowptr, P.col, P.val, res_coarse);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

extern "C" int saena_b200_set_fused_restrict(saena_b200_ctx *ctx, int levels) {
    if (!ctx) return 1;
    ctx->fused_restrict_levels = levels < 0 ? 0 : levels;
    sb_invalidate_graphs(ctx);
    return 0;
}

extern "C" int saena_b200_time_residual_restrict(saena_b200_ctx *ctx, int level, const double *u_host, const double *rhs_host,
                                                 int reps, float *ms_two_kernels, float *ms_fused, double *rel_diff) {
    if (!ctx) return 1;
    SB_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->finalized) SB_FAIL("call saena_b200_finalize first");
    if (ctx->nranks != 1) SB_FAIL("time_residual_restrict: one rank (a measurement)");
    if (level < 0 || level + 1 >= (int)ctx->levels.size()) SB_FAIL("time_residual_restrict: no such level");
    DevLevel &lv = ctx->levels[level];
    DevOperator &A = lv.A, &P = lv.P, &R = lv.R;
    if (A.mapping != SB_MAPPING_SELL || !A.sell.ptr) SB_FAIL("time_residual_restrict: A of this level is not on the sliced layout");
    if (!P.present || P.wide_offsets || !P.col || !P.val) SB_FAIL("time_residual_restrict: P needs 32-bit CSR arrays");
    if (reps < 3) reps = 10;
    const int M = lv.M, Mc = R.M;
    double *u = nullptr, *rhs = nullptr, *out1 = nullptr, *out2 = nullptr;
    SB_CUDA(cudaMalloc((void **)&u, sizeof(double) * M));
    SB_CUDA(cudaMalloc((void **)&rhs, sizeof(double) * M));
    SB_CUDA(cudaMalloc((void **)&out1, sizeof(double) * std::max(Mc, 1)));
    SB_CUDA(cudaMalloc((void **)&out2, sizeof(double) * std::max(Mc, 1)));
    SB_CUDA(cudaMemcpy(u, u_host, sizeof(double) * M, cudaMemcpyHostToDevice));
    SB_CUDA(cudaMemcpy(rhs, rhs_host, sizeof(double) * M, cudaMemcpyHostToDevice));
    cudaStream_t s = ctx->stream;
    auto median = [](std::vector<float> &t) { std::sort(t.begin(), t.end()); return t[t.size() / 2]; };
    int rc = 0;
    std::vector<float> t1, t2;
    for (int it = -2; it < reps && !rc; ++it) {
        // ---- the solve path's two kernels: residual (fused epilogue of the SpMV), then R
        cudaEventRecord(ctx->ev_t0, s);
        EpiArgs e{};
        e.rhs = rhs;
        e.out = lv.res;
        rc = sb_apply(ctx, A, u, EPI_RESIDUAL, e);
        EpiArgs e2{};
        e2.out = out1;
        if (!rc) rc = sb_apply(ctx, R, lv.res, EPI_PLAIN, e2);
        cudaEventRecord(ctx->ev_t1, s);
        cudaEventSynchronize(ctx->ev_t1);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ctx->ev_t0, ctx->ev_t1);
        if (it >= 0) t1.push_back(ms);
        // ---- fused: zero-fill of the coarse vector + one kernel that never writes res
        cudaEventRecord(ctx->ev_t0, s);
        cudaMemsetAsync(out2, 0, sizeof(double) * std::max(Mc, 1), s);
        residual_restrict_sell_kernel<<<(M + 255) / 256, 256, 0, s>>>(M, A.sell.ptr, A.sell.col, A.sell.val, u, rhs,
                                                                    (const int *)P.rowptr, P.col, P.val, out2);
        cudaEventRecord(ctx->ev_t1, s);
        cudaEventSynchronize(ctx->ev_t1);
        cudaEventElapsedTime(&ms, ctx->ev_t0, ctx->ev_t1);
        if (it >= 0) t2.push_back(ms);
    }
    if (!rc && cudaGetLastError() != cudaSuccess) { ctx->error = "time_residual_restrict: a kernel failed"; rc = 1; }
    if (!rc) {
        *ms_two_kernels = median(t1);
        *ms_fused = median(t2);
        std::vector<double> h1(Mc), h2(Mc);
        cudaMemcpy(h1.data(), out1, sizeof(double) * Mc, cudaMemcpyDeviceToHost);
        cudaMemcpy(h2.data(), out2, sizeof(double) * Mc, cudaMemcpyDeviceToHost);
        double num = 0.0, den = 0.0;
        for (int i = 0; i < Mc; ++i) { num += (h1[i] - h2[i]) * (h1[i] - h2[i]); den += h1[i] * h1[i]; }
        *rel_diff = den > 0.0 ? sqrt(num / den) : sqrt(num);
    }
    cudaFree(u); cudaFree(rhs); cudaFree(out1); cudaFree(out2);
    return rc;
}
