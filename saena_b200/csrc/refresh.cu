// refresh.cu -- saena_b200_update_values: new values for level 0's operator on its uploaded pattern, and every coarse
// operator recomputed as R_l (A_l P_l) on the pattern the setup stored for it (SURVEY.md 8f #4, the lazy update).
//
// A user who solves many systems with one matrix pattern (time steps, Newton steps, coefficient sweeps) keeps the
// aggregates, P and R, every stored pattern, the kernel mappings and row blocks; only values are recomputed.  The
// reference's own update1/2/3 are compiled out (#if 0), so the rule is the setup's: C = R A P is mapped onto the
// stored A_{l+1} the way saena_object::filter (sa_setup_dist.filter_entries_dist) made that pattern --
//   - a stored entry takes C's value;
//   - an off-diagonal entry of C outside the pattern is lumped into its row's diagonal;
//   - a diagonal whose magnitude ends below ALMOST_ZERO, or that C lacks, is 1 (C lacking it: the row's lumped entries
//     are dropped, as the filter drops them);
//   - a stored off-diagonal that C does not contain means A_{l+1} is not a Galerkin product of the level above.
// With the uploaded values this reproduces the setup's own A_{l+1}: the entries outside the pattern are the ones the
// filter lumped.  ||C - C|pattern||_F / ||C||_F per level tells how far the frozen pattern has drifted.
//
// Products: saena_b200_spgemm_symbolic / _numeric (spgemm.cu) on the legacy default stream; everything else on the
// context's non-blocking compute stream, so the two are joined by explicit synchronisations.  The SpGEMM operands need
// 64-bit row offsets: operators with 32-bit ones are widened into temporaries; A P and C are freed after each level.
#include <math.h>

#include <chrono>
#include <string>
#include <vector>

#include "common.h"

namespace {

const double ALMOST_ZERO = 1e-14;   // include/data_struct.h:41 of the reference (sa_setup.ALMOST_ZERO)

enum {
    RF_BAD_DIAG = 1,    // a row without a diagonal entry, or |a_ii| < ALMOST_ZERO
    RF_UNSORTED = 2,    // a stored row whose columns do not ascend (the pattern map searches them)
    RF_MISSING = 4,     // a stored off-diagonal entry that R A P does not contain
    RF_NO_DIAG = 8,     // a stored coarse row without a diagonal entry
};

// phases of update_ms (saena_b200_update_values_times)
enum { T_PRODUCTS = 0, T_MAP = 1, T_LAYOUTS = 2, T_EIG = 3, T_COARSEST = 4 };

__device__ __forceinline__ double rf_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ long long rf_warp_sum(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__global__ void rf_widen_kernel(int n, const int *__restrict__ in, int64_t *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i];
}

// warp per row (one rank: the diagonal is local column == row): flags a row without a diagonal or with
// |a_ii| < ALMOST_ZERO (the setup's "zero diagonal element"), and writes inv_diag = 1 / a_ii where asked
template <typename OffT>
__global__ void rf_diag_kernel(int M, const OffT *__restrict__ rowptr, const int *__restrict__ col,
                               const double *__restrict__ val, double *__restrict__ inv_diag, int *__restrict__ flags) {
    const long long gt = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int row = (int)(gt >> 5), lane = threadIdx.x & 31;
    if (row >= M) return;
    double d = 0.0;
    long long found = 0;
    for (long long k = (long long)rowptr[row] + lane; k < (long long)rowptr[row + 1]; k += 32)
        if (col[k] == row) { d += val[k]; ++found; }
    d = rf_warp_sum(d);
    found = rf_warp_sum(found);
    if (lane) return;
    if (!found || !(fabs(d) >= ALMOST_ZERO)) atomicOr(flags, RF_BAD_DIAG);
    if (inv_diag) inv_diag[row] = 1.0 / d;
}

// warp per row: every stored row's columns strictly ascend
template <typename OffT>
__global__ void rf_sorted_kernel(int M, const OffT *__restrict__ rowptr, const int *__restrict__ col,
                                 int *__restrict__ flags) {
    const long long gt = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int row = (int)(gt >> 5), lane = threadIdx.x & 31;
    if (row >= M) return;
    const long long b = (long long)rowptr[row + 1];
    for (long long k = (long long)rowptr[row] + lane; k + 1 < b; k += 32)
        if (col[k] >= col[k + 1]) { atomicOr(flags, RF_UNSORTED); return; }
}

// C = R A P mapped onto the stored pattern of A_{l+1}, one warp per row: C's row ascends; each of its columns is found
// in the stored row by binary search.  norms[0] += ||C||_F^2, norms[1] += the lumped entries' ||.||_F^2.
template <typename OffT>
__global__ void rf_map_kernel(int M, const OffT *__restrict__ rowptr, const int *__restrict__ scol,
                              double *__restrict__ sval, const int64_t *__restrict__ crp, const int *__restrict__ ccol,
                              const double *__restrict__ cval, int *__restrict__ flags, double *__restrict__ norms) {
    const long long gt = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int row = (int)(gt >> 5), lane = threadIdx.x & 31;
    if (row >= M) return;
    const long long s0 = (long long)rowptr[row], s1 = (long long)rowptr[row + 1];
    double cdiag = 0.0, lump = 0.0, lump_sq = 0.0, c_sq = 0.0;
    long long matched = 0, has_cdiag = 0, dpos = -1;
    for (long long k = crp[row] + lane; k < crp[row + 1]; k += 32) {
        const int c = ccol[k];
        const double v = cval[k];
        c_sq += v * v;
        if (c == row) { cdiag += v; has_cdiag = 1; continue; }
        long long lo = s0, hi = s1;
        while (lo < hi) {
            const long long mid = lo + ((hi - lo) >> 1);
            if (scol[mid] < c) lo = mid + 1; else hi = mid;
        }
        if (lo < s1 && scol[lo] == c) {
            sval[lo] = v;
            ++matched;
        } else {
            lump += v;
            lump_sq += v * v;
        }
    }
    for (long long k = s0 + lane; k < s1; k += 32)
        if (scol[k] == row) dpos = k;
    cdiag = rf_warp_sum(cdiag);
    lump = rf_warp_sum(lump);
    lump_sq = rf_warp_sum(lump_sq);
    c_sq = rf_warp_sum(c_sq);
    matched = rf_warp_sum(matched);
    has_cdiag = rf_warp_sum(has_cdiag);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dpos = max(dpos, (long long)__shfl_xor_sync(0xffffffffu, dpos, o));
    if (lane) return;
    if (dpos < 0) {
        atomicOr(flags, RF_NO_DIAG);
    } else {
        double d = has_cdiag ? cdiag + lump : 1.0;
        if (fabs(d) < ALMOST_ZERO) d = 1.0;
        sval[dpos] = d;
    }
    if (matched != (s1 - s0) - (dpos >= 0 ? 1 : 0)) atomicOr(flags, RF_MISSING);
    atomicAdd(&norms[0], c_sq);
    atomicAdd(&norms[1], lump_sq);
}

int warp_blocks(int rows) { return (int)(((long long)rows * 32 + 255) / 256); }

template <typename OffT>
void launch_diag(saena_b200_ctx *ctx, const DevOperator &op, const double *val, double *inv_diag, int *flags) {
    if (op.M)
        rf_diag_kernel<OffT><<<warp_blocks(op.M), 256, 0, ctx->stream>>>(op.M, (const OffT *)op.rowptr, op.col, val,
                                                                          inv_diag, flags);
}

void diag(saena_b200_ctx *ctx, const DevOperator &op, const double *val, double *inv_diag, int *flags) {
    if (op.wide_offsets) launch_diag<int64_t>(ctx, op, val, inv_diag, flags);
    else launch_diag<int>(ctx, op, val, inv_diag, flags);
}

// device buffers of one scope, released on every way out
struct Temps {
    std::vector<void *> p;
    ~Temps() { release(); }
    void release() {
        for (void *q : p) cudaFree(q);
        p.clear();
    }
    template <typename T>
    cudaError_t alloc(T **out, size_t n) {
        *out = nullptr;
        const cudaError_t e = cudaMalloc((void **)out, sizeof(T) * (n ? n : 1));
        if (e == cudaSuccess) p.push_back(*out);
        return e;
    }
};

// the operator's row offsets as int64 (the SpGEMM's operand format): its own array, or a widened temporary
int rowptr64(saena_b200_ctx *ctx, const DevOperator &op, Temps &t, const int64_t **out) {
    if (op.wide_offsets) {
        *out = (const int64_t *)op.rowptr;
        return 0;
    }
    int64_t *w = nullptr;
    SB_CUDA(t.alloc(&w, (size_t)op.M + 1));
    rf_widen_kernel<<<(op.M + 1 + 255) / 256, 256, 0, ctx->stream>>>(op.M + 1, (const int *)op.rowptr, w);
    SB_CUDA(cudaGetLastError());
    *out = w;
    return 0;
}

int spgemm_failed(saena_b200_ctx *ctx, int l) {
    ctx->error = "update_values: level " + std::to_string(l) + " product: " + g_sb_init_error;
    return 1;
}

// C = R_l (A_l P_l) of level l, mapped onto A_{l+1}'s stored values; lumped fraction in *dropped
int refresh_level(saena_b200_ctx *ctx, int l, int *flags_dev, double *norms_dev, double *dropped, double *ms) {
    DevLevel &lv = ctx->levels[l];
    DevOperator &A = lv.A, &P = lv.P, &R = lv.R, &Ac = ctx->levels[l + 1].A;
    auto t0 = std::chrono::steady_clock::now();
    Temps t;
    const int64_t *a_rp = nullptr, *p_rp = nullptr, *r_rp = nullptr;
    SB_TRY(rowptr64(ctx, A, t, &a_rp));
    SB_TRY(rowptr64(ctx, P, t, &p_rp));
    SB_TRY(rowptr64(ctx, R, t, &r_rp));
    // A's values were written and the widened offsets made on the compute stream; the products read them from the
    // default stream, which does not wait for a non-blocking stream
    SB_TRY(sb_sync_stream(ctx, ctx->stream));
    const int M = A.M, Mc = lv.M_coarse_old;
    Temps prod;
    int64_t *ap_rp = nullptr, *c_rp = nullptr;
    int *ap_col = nullptr, *c_col = nullptr;
    double *ap_val = nullptr, *c_val = nullptr;
    int64_t nnz_ap = 0, nnz_c = 0;
    SB_CUDA(prod.alloc(&ap_rp, (size_t)M + 1));
    if (saena_b200_spgemm_symbolic(M, A.n_local_cols, Mc, a_rp, A.col, p_rp, P.col, ap_rp, &nnz_ap)) return spgemm_failed(ctx, l);
    SB_CUDA(prod.alloc(&ap_col, (size_t)nnz_ap));
    SB_CUDA(prod.alloc(&ap_val, (size_t)nnz_ap));
    if (saena_b200_spgemm_numeric(M, A.n_local_cols, Mc, a_rp, A.col, A.val, p_rp, P.col, P.val, ap_rp, ap_col, ap_val))
        return spgemm_failed(ctx, l);
    Temps c;
    SB_CUDA(c.alloc(&c_rp, (size_t)Mc + 1));
    if (saena_b200_spgemm_symbolic(Mc, M, Mc, r_rp, R.col, ap_rp, ap_col, c_rp, &nnz_c)) return spgemm_failed(ctx, l);
    SB_CUDA(c.alloc(&c_col, (size_t)nnz_c));
    SB_CUDA(c.alloc(&c_val, (size_t)nnz_c));
    if (saena_b200_spgemm_numeric(Mc, M, Mc, r_rp, R.col, R.val, ap_rp, ap_col, ap_val, c_rp, c_col, c_val))
        return spgemm_failed(ctx, l);
    prod.release();
    t.release();
    SB_CUDA(cudaStreamSynchronize(cudaStreamLegacy));   // C is complete before a compute-stream kernel reads it
    auto t1 = std::chrono::steady_clock::now();

    SB_CUDA(cudaMemsetAsync(flags_dev, 0, sizeof(int), ctx->stream));
    SB_CUDA(cudaMemsetAsync(norms_dev, 0, 2 * sizeof(double), ctx->stream));
    if (Mc) {
        if (Ac.wide_offsets)
            rf_map_kernel<int64_t><<<warp_blocks(Mc), 256, 0, ctx->stream>>>(Mc, (const int64_t *)Ac.rowptr, Ac.col, Ac.val,
                                                                              c_rp, c_col, c_val, flags_dev, norms_dev);
        else
            rf_map_kernel<int><<<warp_blocks(Mc), 256, 0, ctx->stream>>>(Mc, (const int *)Ac.rowptr, Ac.col, Ac.val, c_rp,
                                                                          c_col, c_val, flags_dev, norms_dev);
    }
    diag(ctx, Ac, Ac.val, ctx->levels[l + 1].inv_diag, flags_dev);
    SB_CUDA(cudaGetLastError());
    int flags = 0;
    double norms[2] = {0.0, 0.0};
    SB_CUDA(cudaMemcpyAsync(&flags, flags_dev, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaMemcpyAsync(norms, norms_dev, sizeof(norms), cudaMemcpyDeviceToHost, ctx->stream));
    SB_TRY(sb_sync_stream(ctx, ctx->stream));
    c.release();
    auto t2 = std::chrono::steady_clock::now();
    ms[T_PRODUCTS] += std::chrono::duration<double, std::milli>(t1 - t0).count();
    ms[T_MAP] += std::chrono::duration<double, std::milli>(t2 - t1).count();
    const std::string where = "update_values: level " + std::to_string(l + 1) + ": ";
    if (flags & RF_MISSING)
        SB_FAIL(where + "A_" + std::to_string(l + 1) + " is not a Galerkin product of the level above (a stored "
                "off-diagonal entry is not in R A P)");
    if (flags & RF_NO_DIAG) SB_FAIL(where + "a stored row has no diagonal entry");
    if (flags & RF_BAD_DIAG) SB_FAIL(where + "a diagonal entry is not finite");
    *dropped = norms[0] > 0.0 ? sqrt(norms[1] / norms[0]) : 0.0;
    return 0;
}

// every check that can refuse the update, before anything is written
int update_refusal(saena_b200_ctx *ctx, const double *val_dev, int64_t nnz, int *flags_dev) {
    if (ctx->nranks > 1)
        SB_FAIL("update_values: one rank only: the coarse product of a row-partitioned level needs the other ranks' "
                "rows of P");
    if (ctx->scale) SB_FAIL("update_values: not on a scaled hierarchy (scale=true)");
    const int L = (int)ctx->levels.size();
    const DevOperator &a0 = ctx->levels[0].A;
    if (nnz != a0.nnz_local)
        SB_FAIL("update_values: nnz_local " + std::to_string(nnz) + " differs from level 0's uploaded " +
                std::to_string(a0.nnz_local));
    for (int l = 0; l < L; ++l) {
        const DevLevel &lv = ctx->levels[l];
        if (lv.A.sell_only)
            SB_FAIL("update_values: level " + std::to_string(l) + "'s operator kept only its sliced copy "
                    "(sliced_only): its CSR values were released");
        if (l + 1 < L && !lv.repart.identity())
            SB_FAIL("update_values: level " + std::to_string(l) + " repartitions its coarse vector");
    }
    SB_CUDA(cudaMemsetAsync(flags_dev, 0, sizeof(int), ctx->stream));
    diag(ctx, a0, val_dev, nullptr, flags_dev);   // on the new values: the setup's zero-diagonal check
    for (int l = 1; l < L; ++l) {
        const DevOperator &A = ctx->levels[l].A;
        if (!A.M) continue;
        if (A.wide_offsets)
            rf_sorted_kernel<int64_t><<<warp_blocks(A.M), 256, 0, ctx->stream>>>(A.M, (const int64_t *)A.rowptr, A.col,
                                                                                 flags_dev);
        else
            rf_sorted_kernel<int><<<warp_blocks(A.M), 256, 0, ctx->stream>>>(A.M, (const int *)A.rowptr, A.col, flags_dev);
    }
    SB_CUDA(cudaGetLastError());
    int flags = 0;
    SB_CUDA(cudaMemcpyAsync(&flags, flags_dev, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    SB_TRY(sb_sync_stream(ctx, ctx->stream));
    if (flags & RF_BAD_DIAG)
        SB_FAIL("update_values: zero diagonal element in the new level-0 values (missing, or |a_ii| < 1e-14)");
    if (flags & RF_UNSORTED)
        SB_FAIL("update_values: a stored coarse operator has a row whose columns do not ascend");
    return 0;
}

// the coarsest level's CSR, downloaded, as the global COO the dense factor is made from
int refactor_coarsest(saena_b200_ctx *ctx) {
    const DevOperator &A = ctx->levels.back().A;
    const int n = A.M;
    std::vector<int64_t> rp((size_t)n + 1);
    if (A.wide_offsets) {
        SB_CUDA(cudaMemcpy(rp.data(), A.rowptr, sizeof(int64_t) * rp.size(), cudaMemcpyDeviceToHost));
    } else {
        std::vector<int> rp32(rp.size());
        SB_CUDA(cudaMemcpy(rp32.data(), A.rowptr, sizeof(int) * rp32.size(), cudaMemcpyDeviceToHost));
        std::copy(rp32.begin(), rp32.end(), rp.begin());
    }
    const int64_t nnz = rp[n];
    std::vector<int32_t> row((size_t)nnz), col((size_t)nnz);
    std::vector<double> val((size_t)nnz);
    SB_CUDA(cudaMemcpy(col.data(), A.col, sizeof(int) * nnz, cudaMemcpyDeviceToHost));
    SB_CUDA(cudaMemcpy(val.data(), A.val, sizeof(double) * nnz, cudaMemcpyDeviceToHost));
    for (int i = 0; i < n; ++i)
        for (int64_t k = rp[i]; k < rp[i + 1]; ++k) row[k] = i;
    return sb_coarsest_factor(ctx, n, nnz, row.data(), col.data(), val.data());
}

// everything after the checks: writes, so a failure leaves the hierarchy half-updated
int update_body(saena_b200_ctx *ctx, const double *val_dev, int64_t nnz, int max_eig_iter, unsigned long long seed,
                double *dropped, int *flags_dev, double *norms_dev) {
    using clk = std::chrono::steady_clock;
    double *ms = ctx->update_ms;
    const int L = (int)ctx->levels.size();
    sb_invalidate_graphs(ctx);   // a captured V-cycle carries the old Chebyshev constants
    // level 0: the values, its diagonal
    auto t0 = clk::now();
    DevLevel &l0 = ctx->levels[0];
    if (nnz) SB_CUDA(cudaMemcpyAsync(l0.A.val, val_dev, sizeof(double) * nnz, cudaMemcpyDeviceToDevice, ctx->stream));
    diag(ctx, l0.A, l0.A.val, l0.inv_diag, flags_dev);
    SB_CUDA(cudaGetLastError());
    ms[T_MAP] += std::chrono::duration<double, std::milli>(clk::now() - t0).count();
    // every coarse level from the one above
    dropped[0] = 0.0;
    for (int l = 0; l + 1 < L; ++l) SB_TRY(refresh_level(ctx, l, flags_dev, norms_dev, &dropped[l + 1], ms));
    // the sliced copies of the entries (the eigenvalue estimate and the route probe apply the operators through them)
    auto t1 = clk::now();
    // the symmetric diagonals are filled and checked again; an operator whose new values are not symmetric moves to the
    // sliced layout here, before anything applies it
    for (DevLevel &lv : ctx->levels) {
        if (lv.A.sell.ptr) SB_TRY(sb_fill_sliced(ctx, lv.A, lv.A.sell));
        if (lv.A.sellp.ptr) SB_TRY(sb_fill_sliced(ctx, lv.A, lv.A.sellp));
        SB_TRY(sb_refresh_symdiag(ctx, lv.A));
    }
    auto t2 = clk::now();
    for (int l = 0; l < L; ++l) {   // find_eig(store = 1) on every level
        double e = 0.0;
        SB_TRY(sb_find_eig(ctx, l, max_eig_iter, nullptr, seed, &e, nullptr));
        ctx->levels[l].eig_max = e;
    }
    auto t3 = clk::now();
    if (ctx->coarse_n > 0) SB_TRY(refactor_coarsest(ctx));
    auto t4 = clk::now();
    ms[T_LAYOUTS] += std::chrono::duration<double, std::milli>(t2 - t1).count();
    ms[T_EIG] += std::chrono::duration<double, std::milli>(t3 - t2).count();
    ms[T_COARSEST] += std::chrono::duration<double, std::milli>(t4 - t3).count();
    sb_invalidate_graphs(ctx);
    return sb_recheck_routes(ctx);
}

}  // namespace

int sb_update_values(saena_b200_ctx *ctx, const double *val_dev, int64_t nnz, int max_eig_iter, unsigned long long seed,
                     double *dropped_out, int dropped_cap) {
    for (double &m : ctx->update_ms) m = 0.0;
    Temps t;
    int *flags_dev = nullptr;
    double *norms_dev = nullptr;
    SB_CUDA(t.alloc(&flags_dev, 1));
    SB_CUDA(t.alloc(&norms_dev, 2));
    SB_TRY(update_refusal(ctx, val_dev, nnz, flags_dev));
    std::vector<double> dropped(ctx->levels.size(), 0.0);
    if (update_body(ctx, val_dev, nnz, max_eig_iter, seed, dropped.data(), flags_dev, norms_dev)) {
        ctx->finalized = false;
        ctx->error += " -- the hierarchy is half-updated: upload it again";
        return 1;
    }
    for (int i = 0; dropped_out && i < dropped_cap && i < (int)dropped.size(); ++i) dropped_out[i] = dropped[i];
    return 0;
}
