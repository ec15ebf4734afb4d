// fused_halo.cu -- the distributed SpMV of one rank as ONE kernel: ghost-value exchange over
// NVLink peer memory + interior rows + rows that need ghost values, with the smoother / residual /
// correction epilogue fused as everywhere else.
//
// What it replaces: saena_matrix::matvec_sparse[_float] in full
// (/root/reference/src/saena_matrix_matvec.cpp:9-113, :448-550) -- pack (:25-26), MPI_Isend/Irecv
// (:32-41), local loop (:68-80), MPI_Waitany + remote loop (:87-110) -- and the same structure of
// prolong_matrix::matvec_sparse / restrict_matrix::matvec_sparse.
//
// Why one kernel.  With the exchange as separate launches (pack kernel on a comm stream, stream
// memory-op waits, boundary kernel, signal kernel: p2p_halo.cu) every operator application of a
// multi-rank V-cycle carries ~40 us that no bandwidth explains (measured on 8 B200: 256^3 Poisson,
// levels 2-4, 9 applications per level per V-cycle; replaying the V-cycle from a CUDA graph did
// not remove it, so it is device-side dependency latency, not launch cost).  Here a CTA's role
// follows from its index:
//
//   [0, n_pack)                  pack: gather x[vIndex[i]] (rounded through float when the operator's
//                                use_double is false -- the same value matvec_sparse_float widens
//                                on the receiving side) and store it straight into the receiving
//                                rank's landing area; the last pack CTA raises `arrived` there
//   [n_pack, n_pack + n_int)     interior rows: no ghost column, start at once -- this is the part
//                                of the SpMV that hides the transfer
//   the rest                     rows with ghost columns: spin (one thread per sender, on this
//                                rank's OWN memory) until `arrived`, then compute.  Split operators
//                                run the boundary-row body (local CSR segment + ghost segment);
//                                merged operators (every row couples to ghosts) run the ordinary
//                                mapping over [local | ghost] columns, the gather choosing the
//                                source by column index -- no x_ext copy, no widen pass.
//   last CTA of each role        raises the flags of the hand-shake and advances the role's counter
//
// The kernel's MAP is the operator's mapping code (DevOperator::mapping), dispatched by the same
// sb_dispatch_mapping as the stand-alone launches and with the same grid rule, sb_mapping_blocks.
//
// The hand-shake (halo_sync.cuh) is shared with the separate-launch form (p2p_halo.cu): monotonic
// counters in device memory, two landing buffers selected by the application's parity, every wait
// bounded by a globaltimer deadline.  A launch carries no host-side state: the kernel replays from
// a CUDA graph.  Progress: CTAs are dispatched in index order, so the pack CTAs of a launch are
// resident before any CTA of the same launch spins; with two buffers they wait only for a
// `consumed` signal the peers sent a whole application earlier.  A waiting CTA's producer is always a
// pack CTA of ANOTHER rank's launch of the same operator, and nothing of this rank stands between
// that launch and the GPU: every earlier launch of this rank has completed (stream order; the
// separate-launch form joins its comm stream before its boundary kernel).  No cycle.
#include <algorithm>

#include "halo_sync.cuh"
#include "spmv_kernels.cuh"

struct FusedArgs {
    // operator (32-bit row offsets only; nnz >= 2^31 keeps the unfused path)
    const int *rowptr;
    const int *col;
    const double *val;
    const long long *sell_ptr;
    const int *sell_col;
    const double *sell_val;
    int M, int_lo, int_hi, n_local;
    // rows with remote entries of a split operator
    int n_brows, bnd_wide;
    const int *brow;
    const int *brow_ptr;
    const int *bcol;
    const double *bval;
    const double *x;
    const double *ghost;  // this rank's landing area: 2 x recvSize doubles
    int recvSize;
    // merged operators on a CSR mapping: rows are stored [local columns | ghost columns], rowmid[i] is where the ghost
    // part of row i starts.  The local part is summed BEFORE the wait (partial[] keeps it), the ghost part after:
    // the exchange hides behind the rows' own local work -- the reference's order too (local loop, then remote loop)
    const int *rowmid;
    double *partial;
    int split;
    EpiArgs e;
    // CTA roles: pack | interior rows | rows that wait for ghosts.  The waiting CTAs are at most a
    // chip-full (resident all at once) and stride over n_wait_blocks virtual blocks, so the
    // hand-shake is paid once per CTA, not once per row block
    int n_pack, n_int, n_wait, n_wait_blocks;
    int do_sync, do_compute;
    // pack
    int vIndexSize, round_float;
    const int *vIndex;
    HaloSync h;
};

template <int MAP, int EPI, typename XS>
__device__ __forceinline__ void fused_rows(int vb, int lo, int hi, const FusedArgs &a, const XS xs) {
    if constexpr (MAP == SB_MAPPING_SELL)
        spmv_sell_body<EPI, XS, 4>(vb, lo, hi, a.sell_ptr, a.sell_col, a.sell_val, xs, a.e, nullptr);
    else if constexpr (MAP >= 32)
        spmv_rowgroup_body<MAP, EPI, int>(vb, lo, hi, a.rowptr, a.col, a.val, xs, a.e, nullptr);
    else
        spmv_vec_body<MAP, EPI, int>(vb, lo, hi, a.rowptr, a.col, a.val, xs, a.e, nullptr);
}

// ---- merged operators, two phases around the wait (PHASE 0: local columns -> partial[], PHASE 1: ghost columns +
//      partial[] -> epilogue).  The thread that finishes a row is the same in both phases (same vb, same mapping), so
//      partial[row] is written and read by one thread: no fence between the phases.
template <int TPR, int EPI, int PHASE>
__device__ __forceinline__ void
fused_rowgroup_phase(int vb, const FusedArgs &a, const double *__restrict__ src) {
    constexpr int ROWS = 256 / TPR;
    constexpr int WPR = TPR / 32;
    __shared__ double s_part2[8];
    const int g = threadIdx.x / TPR, sub = threadIdx.x % TPR;
    const int row = vb * ROWS + g;
    double sum = 0.0;
    if (row < a.M) {
        const int start = PHASE == 0 ? a.rowptr[row] : a.rowmid[row];
        const int end = PHASE == 0 ? a.rowmid[row] : a.rowptr[row + 1];
        for (int k = start + sub; k < end; k += TPR * VEC_UNROLL) {
            int c[VEC_UNROLL];
            double v[VEC_UNROLL];
#pragma unroll
            for (int q = 0; q < VEC_UNROLL; ++q) {
                const int kk = k + q * TPR;
                const bool in = kk < end;
                c[q] = in ? sb_ld_stream(a.col + kk) : (PHASE == 0 ? 0 : a.n_local);
                v[q] = in ? sb_ld_stream(a.val + kk) : 0.0;
            }
#pragma unroll
            for (int q = 0; q < VEC_UNROLL; ++q) sum += v[q] * (PHASE == 0 ? __ldg(src + c[q]) : src[c[q] - a.n_local]);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (WPR > 1) {
        if ((threadIdx.x & 31) == 0) s_part2[threadIdx.x >> 5] = sum;
        __syncthreads();
        if (sub == 0) {
            sum = 0.0;
#pragma unroll
            for (int w = 0; w < WPR; ++w) sum += s_part2[g * WPR + w];
        }
    }
    if (sub == 0 && row < a.M) {
        if (PHASE == 0) a.partial[row] = sum;
        else sb_epilogue<EPI>(row, a.partial[row] + sum, a.e);
    }
    if (WPR > 1) __syncthreads();  // s_part2 is reused by the next virtual block
}

template <int LANES, int EPI, int PHASE>
__device__ __forceinline__ void
fused_vec_phase(int vb, const FusedArgs &a, const double *__restrict__ src) {
    constexpr int G = 32 / LANES;
    const int lane = threadIdx.x & 31;
    const int warp = (vb * 256 + threadIdx.x) >> 5;
    const int row0 = warp * 32;
    if (row0 >= a.M) return;
    const int my_row = row0 + lane;
    int my_start = 0, my_end = 0;
    if (my_row < a.M) {
        my_start = PHASE == 0 ? a.rowptr[my_row] : a.rowmid[my_row];
        my_end = PHASE == 0 ? a.rowmid[my_row] : a.rowptr[my_row + 1];
    }
    double mine = 0.0;
    const int g = lane / LANES, sub = lane % LANES;
#pragma unroll
    for (int t = 0; t < LANES; ++t) {
        const int srcl = t * G + g;
        const int start = __shfl_sync(0xffffffffu, my_start, srcl);
        const int end = __shfl_sync(0xffffffffu, my_end, srcl);
        double sum = 0.0;
        for (int k = start + sub; k < end; k += LANES * VEC_UNROLL) {
            int c[VEC_UNROLL];
            double v[VEC_UNROLL];
#pragma unroll
            for (int q = 0; q < VEC_UNROLL; ++q) {
                const int kk = k + q * LANES;
                const bool in = kk < end;
                c[q] = in ? sb_ld_stream(a.col + kk) : (PHASE == 0 ? 0 : a.n_local);
                v[q] = in ? sb_ld_stream(a.val + kk) : 0.0;
            }
#pragma unroll
            for (int q = 0; q < VEC_UNROLL; ++q) sum += v[q] * (PHASE == 0 ? __ldg(src + c[q]) : src[c[q] - a.n_local]);
        }
#pragma unroll
        for (int o = LANES / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        const double v = __shfl_sync(0xffffffffu, sum, (lane % G) * LANES);
        if (lane / G == t) mine = v;
    }
    if (my_row < a.M) {
        if (PHASE == 0) a.partial[my_row] = mine;
        else sb_epilogue<EPI>(my_row, a.partial[my_row] + mine, a.e);
    }
}

template <int MAP, int EPI, int PHASE>
__device__ __forceinline__ void fused_rows_phase(int vb, const FusedArgs &a, const double *src) {
    if constexpr (MAP >= 32 && MAP != SB_MAPPING_SELL) fused_rowgroup_phase<MAP, EPI, PHASE>(vb, a, src);
    else if constexpr (MAP != SB_MAPPING_SELL) fused_vec_phase<MAP, EPI, PHASE>(vb, a, src);
}

// The mappings whose stand-alone kernels fit 32 registers keep 8 CTAs per SM here too (the role
// dispatch and the stride loop would otherwise push them to 40 and cost a quarter of the loads in
// flight on the big fine levels); the 4/8/16-lane sub-warp mappings need 40-48 either way.
template <int MAP>
constexpr int fused_min_ctas() { return (MAP == 4 || MAP == 8 || MAP == 16) ? 4 : 8; }

template <int MAP, int EPI, bool MERGED>
__global__ void __launch_bounds__(256, fused_min_ctas<MAP>())
fused_halo_spmv_kernel(const __grid_constant__ FusedArgs a) {
    __shared__ unsigned long long s_epoch;
    const int b = blockIdx.x, tid = threadIdx.x;
    if (b >= a.n_pack && b < a.n_pack + a.n_int) {
        // interior rows of a split operator: nothing to wait for
        fused_rows<MAP, EPI>(b - a.n_pack, a.int_lo, a.int_hi, a, XLocal{a.x});
        return;
    }
    const bool packer = b < a.n_pack;
    if (a.do_sync) {
        if (tid == 0) s_epoch = *(volatile unsigned long long *)&a.h.epoch[packer ? 0 : 1];
        __syncthreads();
    }
    const unsigned long long done = a.do_sync ? s_epoch : 0ull;  // applications this role completed before this one
    if (packer) {
        sb_halo_pack_cta(a.h, b, a.n_pack, done, a.x, a.vIndex, a.vIndexSize, a.round_float != 0);
        return;
    }
    // ---- rows that read ghost values
    if constexpr (MERGED && MAP != SB_MAPPING_SELL) {
        if (a.split) {
            // local columns first: this is what the exchange hides behind on a merged operator
            for (int vb = b - a.n_pack; vb < a.n_wait_blocks; vb += a.n_wait) fused_rows_phase<MAP, EPI, 0>(vb, a, a.x);
            sb_halo_wait_cta(a.h, done);
            const double *ghost = a.ghost + (size_t)(done & 1ull) * (size_t)a.recvSize;
            for (int vb = b - a.n_pack; vb < a.n_wait_blocks; vb += a.n_wait) fused_rows_phase<MAP, EPI, 1>(vb, a, ghost);
            sb_halo_release_cta(a.h, a.n_wait, done);
            return;
        }
    }
    if (a.do_sync) sb_halo_wait_cta(a.h, done);
    if (a.do_compute) {
        const double *ghost = a.ghost + (size_t)(done & 1ull) * (size_t)a.recvSize;
        for (int vb = b - a.n_pack - a.n_int; vb < a.n_wait_blocks; vb += a.n_wait) {
            if constexpr (MERGED) {
                fused_rows<MAP, EPI>(vb, 0, a.M, a, XGhost{a.x, ghost, a.n_local});
                if constexpr (MAP >= 64 && MAP != SB_MAPPING_SELL) __syncthreads();  // s_part is reused
            } else {
                if (a.bnd_wide)
                    spmv_boundary_body<32, EPI, int, double>(vb, a.n_brows, a.brow, a.rowptr, a.col, a.val,
                                                             a.brow_ptr, a.bcol, a.bval, a.x, ghost, a.e);
                else
                    spmv_boundary_body<8, EPI, int, double>(vb, a.n_brows, a.brow, a.rowptr, a.col, a.val,
                                                            a.brow_ptr, a.bcol, a.bval, a.x, ghost, a.e);
            }
        }
    }
    if (a.do_sync) sb_halo_release_cta(a.h, a.n_wait, done);
}

// The fused kernel covers the 32-bit-offset CSR / sliced mappings; anything else (64-bit row offsets, the
// streaming mapping) takes the separate launches, which speak the same hand-shake -- the choice is local.
bool sb_fused_eligible(const DevOperator &op) {
    return op.p2p && op.fused && !op.wide_offsets && op.mapping > 0 && op.mapping != SB_MAPPING_SELLP &&
           op.mapping != SB_MAPPING_SYMDIAG &&
           (!op.sends.empty() || !op.recvs.empty());
}

template <int EPI, bool MERGED>
static int launch_fused(saena_b200_ctx *ctx, const DevOperator &op, const FusedArgs &a, int grid) {
    const bool known = sb_dispatch_mapping(op.mapping, [&](auto map) {
        fused_halo_spmv_kernel<decltype(map)::value, EPI, MERGED><<<grid, 256, 0, ctx->stream>>>(a);
    });
    if (!known) SB_FAIL("fused apply: unknown mapping");
    SB_CUDA(cudaGetLastError());
    return 0;
}

template <int EPI>
static int apply_fused_epi(saena_b200_ctx *ctx, DevOperator &op, const double *x, const EpiArgs &e) {
    const int mode = ctx->apply_mode;  // 0 full, 1 compute only (stale ghosts), 2 exchange only
    FusedArgs a{};
    a.rowptr = (const int *)op.rowptr; a.col = op.col; a.val = op.val;
    a.sell_ptr = op.sell.ptr; a.sell_col = op.sell.col; a.sell_val = op.sell.val;
    a.M = op.M; a.int_lo = op.int_lo; a.int_hi = op.int_hi; a.n_local = op.n_local_cols;
    a.n_brows = op.n_brows; a.bnd_wide = op.avg_nnz_row() >= 48.0;
    a.brow = op.brow; a.brow_ptr = op.brow_ptr; a.bcol = op.bcol; a.bval = op.bval;
    a.x = x; a.ghost = op.ghost_d; a.recvSize = op.recvSize; a.e = e;
    a.rowmid = op.rowmid; a.partial = op.partial;
    a.split = mode == 0 && op.merged && op.mapping != SB_MAPPING_SELL && op.rowmid && op.partial && ctx->merged_split;
    a.do_sync = mode != 1;
    a.do_compute = mode != 2;
    a.vIndexSize = op.vIndexSize; a.vIndex = op.vIndex;
    a.round_float = !op.use_double;
    a.h = sb_halo_sync_args(ctx, op);
    a.n_pack = mode == 1 ? 0 : (op.vIndexSize + SB_PACK_PER_CTA - 1) / SB_PACK_PER_CTA;
    if (op.merged) {
        a.n_int = 0;
        a.n_wait_blocks = sb_mapping_blocks(op.mapping, op.M);
    } else {
        a.n_int = sb_mapping_blocks(op.mapping, op.int_hi - op.int_lo);
        const int rows_per_block = 256 / (a.bnd_wide ? 32 : 8);
        a.n_wait_blocks = (op.n_brows + rows_per_block - 1) / rows_per_block;
    }
    if (mode == 2) {
        a.n_int = 0;
        a.n_wait_blocks = op.recvs.empty() ? 0 : 1;
    }
    // a chip-full of waiting CTAs (8 x 256 threads per SM at <= 32 registers; fewer fit for the
    // wider sub-warp mappings, the excess simply starts later -- every spinning CTA's producer is
    // a pack CTA of another rank, never a CTA behind it in this grid)
    a.n_wait = std::min(a.n_wait_blocks, 8 * ctx->sm_count);
    if (mode != 1 && a.n_wait == 0 && !op.recvs.empty()) SB_FAIL("fused apply: receives but no row reads them");
    if (a.h.n_segs > 256 || a.h.n_recv > 256) SB_FAIL("fused apply: more than 256 neighbours (one spinning thread each)");
    const int grid = a.n_pack + a.n_int + a.n_wait;
    if (grid == 0) return 0;
    ++ctx->launches;
    if (op.merged) return launch_fused<EPI, true>(ctx, op, a, grid);
    return launch_fused<EPI, false>(ctx, op, a, grid);
}

int sb_apply_fused(saena_b200_ctx *ctx, DevOperator &op, const double *x, int epi, const EpiArgs &args) {
    switch (epi) {
        case EPI_PLAIN: return apply_fused_epi<EPI_PLAIN>(ctx, op, x, args);
        case EPI_RESIDUAL: return apply_fused_epi<EPI_RESIDUAL>(ctx, op, x, args);
        case EPI_CHEB_FIRST: return apply_fused_epi<EPI_CHEB_FIRST>(ctx, op, x, args);
        case EPI_CHEB_NEXT: return apply_fused_epi<EPI_CHEB_NEXT>(ctx, op, x, args);
        case EPI_JACOBI: return apply_fused_epi<EPI_JACOBI>(ctx, op, x, args);
        case EPI_SUB: return apply_fused_epi<EPI_SUB>(ctx, op, x, args);
    }
    SB_FAIL("fused apply: unknown epilogue");
}
