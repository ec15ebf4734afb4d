// spmv_block.cu -- one operator application to a block of k <= SB_BLOCK_MAX column-major vectors
// (saena_b200_solve_pcg_block and its hooks).  The mappings the hierarchies use -- the sliced layouts 100 / 101, the
// symmetric diagonals 103, spmv_vec and spmv_rowgroup -- stream the operator once for all k columns
// (spmv_kernels.cuh, *_block_kernel).  Everything else -- streaming row blocks, operators with the dense flag, a halo or
// the merged layout -- applies the single kernel to one column after the other through sb_apply, which keeps every
// hierarchy correct without block versions of kernels no benchmarked level runs.
#include "spmv_kernels.cuh"

// column j of a block epilogue: every vector but inv_diag (one per row) offset by j * ld
static EpiArgs epi_column(const EpiArgs &e, int j, long long ld) {
    EpiArgs c = e;
    const long long o = (long long)j * ld;
    if (c.rhs) c.rhs += o;
    if (c.d_in) c.d_in += o;
    if (c.d_out) c.d_out += o;
    if (c.u_in) c.u_in += o;
    if (c.out) c.out += o;
    return c;
}

static bool has_block_body(const saena_b200_ctx *ctx, const DevOperator &op) {
    if (ctx->nranks != 1 || op.merged || !op.sends.empty() || !op.recvs.empty() || op.n_brows) return false;
    if (op.use_dense && !op.use_double) return false;
    const int m = op.mapping;
    return m == SB_MAPPING_SELL || m == SB_MAPPING_SELLP || m == SB_MAPPING_SYMDIAG || (m >= 1 && m <= 256);
}

template <int EPI, int K, typename OffT>
static int launch_block(saena_b200_ctx *ctx, DevOperator &op, int k, const double *x, const EpiArgs &e) {
    const OffT *rp = (const OffT *)op.rowptr;
    cudaStream_t s = ctx->stream;
    const long long ldx = op.n_local_cols, ld = op.M;
    const int lo = op.int_lo, hi = op.int_hi;
    if (hi - lo <= 0) return 0;
    ++ctx->launches;
    if (op.mapping == SB_MAPPING_SYMDIAG) {
        const int blocks = (op.M + 255) / 256;
        const double *d = op.sdiag_val;
        if (op.sdiag.nd <= 4)
            spmv_symdiag_block_kernel<4, EPI, K><<<blocks, 256, 0, s>>>(op.M, k, d, op.sdiag, x, ldx, e, ld);
        else if (op.sdiag.nd <= 8)
            spmv_symdiag_block_kernel<8, EPI, K><<<blocks, 256, 0, s>>>(op.M, k, d, op.sdiag, x, ldx, e, ld);
        else
            spmv_symdiag_block_kernel<SYMDIAG_MAX, EPI, K><<<blocks, 256, 0, s>>>(op.M, k, d, op.sdiag, x, ldx, e, ld);
        return 0;
    }
    if (op.mapping == SB_MAPPING_SELLP) {
        spmv_sellp_block_kernel<EPI, K><<<(op.M + 255) / 256, 256, 0, s>>>(op.M, k, op.sellp.ptr, op.sellp.perm,
                                                                            op.sellp.col, op.sellp.val, x, ldx, e, ld);
        return 0;
    }
    const int blocks = sb_mapping_blocks(op.mapping, hi - lo);
    const bool known = sb_dispatch_mapping(op.mapping, [&](auto map) {
        constexpr int MAP = decltype(map)::value;
        if constexpr (MAP == SB_MAPPING_SELL)
            spmv_sell_block_kernel<EPI, K><<<blocks, 256, 0, s>>>(lo, hi, k, op.sell.ptr, op.sell.col, op.sell.val, x,
                                                                  ldx, e, ld);
        else if constexpr (MAP >= 32)
            spmv_rowgroup_block_kernel<MAP, EPI, K, OffT><<<blocks, 256, 0, s>>>(lo, hi, k, rp, op.col, op.val, x, ldx,
                                                                                 e, ld);
        else
            spmv_vec_block_kernel<MAP, EPI, K, OffT><<<blocks, 256, 0, s>>>(lo, hi, k, rp, op.col, op.val, x, ldx, e,
                                                                            ld);
    });
    if (!known) SB_FAIL("apply_block: unknown mapping");
    return 0;
}

template <int EPI, int K>
static int apply_block_k(saena_b200_ctx *ctx, DevOperator &op, int k, const double *x, const EpiArgs &e) {
    if (op.wide_offsets) SB_TRY((launch_block<EPI, K, int64_t>(ctx, op, k, x, e)));
    else SB_TRY((launch_block<EPI, K, int>(ctx, op, k, x, e)));
    SB_CUDA(cudaGetLastError());
    return 0;
}

template <int EPI>
static int apply_block_epi(saena_b200_ctx *ctx, DevOperator &op, int k, const double *x, const EpiArgs &e) {
    if (k <= 2) return apply_block_k<EPI, 2>(ctx, op, k, x, e);
    if (k <= 4) return apply_block_k<EPI, 4>(ctx, op, k, x, e);
    return apply_block_k<EPI, SB_BLOCK_MAX>(ctx, op, k, x, e);
}

int sb_apply_block(saena_b200_ctx *ctx, DevOperator &op, int k, const double *x, int epi, const EpiArgs &args) {
    if (!op.present) SB_FAIL("apply_block: operator was not uploaded");
    if (k < 1 || k > SB_BLOCK_MAX) SB_FAIL("apply_block: k must be in 1..8");
    if (k == 1) return sb_apply(ctx, op, x, epi, args);
    if (!has_block_body(ctx, op)) {
        for (int j = 0; j < k; ++j)
            SB_TRY(sb_apply(ctx, op, x + (long long)j * op.n_local_cols, epi, epi_column(args, j, op.M)));
        return 0;
    }
    switch (epi) {
        case EPI_PLAIN: return apply_block_epi<EPI_PLAIN>(ctx, op, k, x, args);
        case EPI_RESIDUAL: return apply_block_epi<EPI_RESIDUAL>(ctx, op, k, x, args);
        case EPI_CHEB_FIRST: return apply_block_epi<EPI_CHEB_FIRST>(ctx, op, k, x, args);
        case EPI_CHEB_NEXT: return apply_block_epi<EPI_CHEB_NEXT>(ctx, op, k, x, args);
        case EPI_JACOBI: return apply_block_epi<EPI_JACOBI>(ctx, op, k, x, args);
        case EPI_SUB: return apply_block_epi<EPI_SUB>(ctx, op, k, x, args);
    }
    SB_FAIL("apply_block: unknown epilogue");
}
