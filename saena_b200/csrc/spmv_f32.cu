// spmv_f32.cu -- one operator application on its FP32 copy (the FP32 preconditioner, saena_b200_set_precond_precision).
// The bodies are those of spmv_kernels.cuh instantiated on float: the sliced layouts 100 / 101 with their trip-of-8
// row sum, the symmetric diagonals 103 in their 4 / 8 / 16 buckets, spmv_vec (1..16) and spmv_rowgroup (32..256).  Each
// row is summed in the FP64 kernel's column order with `sum += a * x` in float, and the epilogue runs in float.  The
// operator's FP32 values (sell.val32, sellp.val32, sdiag_val32, val32) share the FP64 layout's column ids, slice
// offsets, permutation and row offsets.  sb_f32_sync refuses every operator without such a body (a halo, the merged
// layout, streaming row blocks), so none reaches this file.  A level with the dense flag runs its mapping's body here:
// its input is float already, the rounding the flag stands for.
#include "spmv_kernels.cuh"

// elementwise conversions: the PCG residual into level 0's FP32 rhs, the V-cycle's result back, the coarsest level's
// vectors around its FP64 solve, and the FP32 copies of the values and inv_diag
template <typename S, typename D>
__global__ void __launch_bounds__(256) convert_kernel(size_t n, const S *__restrict__ src, D *__restrict__ dst) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = (D)src[i];
}

template <typename S, typename D>
static int convert(saena_b200_ctx *ctx, size_t n, const S *src, D *dst) {
    if (n == 0) return 0;
    ++ctx->launches;
    const size_t want = (n + 255) / 256, cap = (size_t)ctx->sm_count * 16;
    convert_kernel<S, D><<<(unsigned)(want < cap ? want : cap), 256, 0, ctx->stream>>>(n, src, dst);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int sb_convert(saena_b200_ctx *ctx, size_t n, const double *src, float *dst) { return convert(ctx, n, src, dst); }
int sb_convert(saena_b200_ctx *ctx, size_t n, const float *src, double *dst) { return convert(ctx, n, src, dst); }

template <int EPI, typename OffT>
static int launch_f32(saena_b200_ctx *ctx, DevOperator &op, const float *x, const EpiArgs32 &e) {
    const OffT *rp = (const OffT *)op.rowptr;
    cudaStream_t s = ctx->stream;
    const int lo = op.int_lo, hi = op.int_hi;   // no halo: every row
    if (hi - lo <= 0) return 0;
    ++ctx->launches;
    if (op.mapping == SB_MAPPING_SYMDIAG) {
        const int blocks = (op.M + 255) / 256;
        const float *d = op.sdiag_val32;
        if (op.sdiag.nd <= 4) spmv_symdiag_kernel<4, EPI, float><<<blocks, 256, 0, s>>>(op.M, d, op.sdiag, x, e);
        else if (op.sdiag.nd <= 8) spmv_symdiag_kernel<8, EPI, float><<<blocks, 256, 0, s>>>(op.M, d, op.sdiag, x, e);
        else spmv_symdiag_kernel<SYMDIAG_MAX, EPI, float><<<blocks, 256, 0, s>>>(op.M, d, op.sdiag, x, e);
        return 0;
    }
    if (op.mapping == SB_MAPPING_SELLP) {
        spmv_sellp_kernel<EPI, float><<<(op.M + 255) / 256, 256, 0, s>>>(op.M, op.sellp.ptr, op.sellp.perm,
                                                                          op.sellp.col, op.sellp.val32, x, e);
        return 0;
    }
    const int blocks = sb_mapping_blocks(op.mapping, hi - lo);
    const bool known = sb_dispatch_mapping(op.mapping, [&](auto map) {
        constexpr int MAP = decltype(map)::value;
        if constexpr (MAP == SB_MAPPING_SELL)
            spmv_sell_kernel<EPI, float><<<blocks, 256, 0, s>>>(lo, hi, op.sell.ptr, op.sell.col, op.sell.val32, x, e,
                                                                nullptr);
        else if constexpr (MAP >= 32)
            spmv_rowgroup_kernel<MAP, EPI, OffT, float><<<blocks, 256, 0, s>>>(lo, hi, rp, op.col, op.val32, x, e,
                                                                               nullptr);
        else
            spmv_vec_kernel<MAP, EPI, OffT, float><<<blocks, 256, 0, s>>>(lo, hi, rp, op.col, op.val32, x, e, nullptr);
    });
    if (!known) SB_FAIL("apply_f32: no FP32 body for this mapping");
    return 0;
}

template <int EPI>
static int apply_f32(saena_b200_ctx *ctx, DevOperator &op, const float *x, const EpiArgs32 &e) {
    if (op.wide_offsets) SB_TRY((launch_f32<EPI, int64_t>(ctx, op, x, e)));
    else SB_TRY((launch_f32<EPI, int>(ctx, op, x, e)));
    SB_CUDA(cudaGetLastError());
    return 0;
}

int sb_apply(saena_b200_ctx *ctx, DevOperator &op, const float *x, int epi, const EpiArgs32 &args) {
    if (!op.present) SB_FAIL("apply_f32: operator was not uploaded");
    switch (epi) {
        case EPI_PLAIN: return apply_f32<EPI_PLAIN>(ctx, op, x, args);
        case EPI_RESIDUAL: return apply_f32<EPI_RESIDUAL>(ctx, op, x, args);
        case EPI_CHEB_FIRST: return apply_f32<EPI_CHEB_FIRST>(ctx, op, x, args);
        case EPI_CHEB_NEXT: return apply_f32<EPI_CHEB_NEXT>(ctx, op, x, args);
        case EPI_JACOBI: return apply_f32<EPI_JACOBI>(ctx, op, x, args);
        case EPI_SUB: return apply_f32<EPI_SUB>(ctx, op, x, args);
    }
    SB_FAIL("apply_f32: unknown epilogue");
}
