// operator.cu -- upload of one operator in the reference layout and its application on the GPU.
//
// Upload contract = the arrays saena_matrix::set_off_on_diagonal leaves behind
// (/root/reference/src/saena_matrix_setup.cpp:793-1098; same for P and R:
// prolong_matrix.cpp:18-378, restrict_matrix.cpp:229-494).  Device layout (DESIGN.md):
//   local block  -> CSR: rowptr (scan of nnzPerRow_local), col made LOCAL (global - col_offset,
//                   the reference's `v_p = v - split[rank]` folded in at upload), val
//   remote block -> re-sorted from column-major-by-sender to row-major over the boundary rows
//                   (no atomics in the remote kernel), column = index into the ghost buffer
//   halo plan    -> vIndex + per-peer (offset,count) slices of the packed send / ghost buffers
#include <algorithm>
#include <climits>
#include <numeric>

#include "spmv_kernels.cuh"

__global__ void localise_cols_kernel(long long n, int *__restrict__ col, int col_offset, int n_local_cols,
                                     int *__restrict__ bad) {
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        const int c = col[k] - col_offset;
        if (c < 0 || c >= n_local_cols) *bad = 1;
        col[k] = c;
    }
}

template <typename T>
static int dev_upload(saena_b200_ctx *ctx, T **dst, const T *src, size_t n) {
    *dst = nullptr;
    SB_CUDA(cudaMalloc((void **)dst, std::max<size_t>(n, 1) * sizeof(T)));
    if (n) SB_CUDA(cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice));
    return 0;
}

// host row offsets -> the operator's rowptr, 64-bit with wide_offsets, else 32-bit
static int upload_rowptr(saena_b200_ctx *ctx, DevOperator &op, const std::vector<int64_t> &rp) {
    if (op.wide_offsets) {
        int64_t *p = nullptr;
        SB_TRY(dev_upload(ctx, &p, rp.data(), rp.size()));
        op.rowptr = p;
    } else {
        std::vector<int> rp32(rp.begin(), rp.end());
        int *p = nullptr;
        SB_TRY(dev_upload(ctx, &p, rp32.data(), rp32.size()));
        op.rowptr = p;
    }
    return 0;
}

// the operator's row offsets back on the host, widened to 64 bits
static int read_rowptr(saena_b200_ctx *ctx, const DevOperator &op, std::vector<int64_t> &rp) {
    rp.assign((size_t)op.M + 1, 0);
    if (op.wide_offsets) {
        SB_CUDA(cudaMemcpy(rp.data(), op.rowptr, sizeof(int64_t) * rp.size(), cudaMemcpyDeviceToHost));
    } else {
        std::vector<int> rp32(rp.size());
        SB_CUDA(cudaMemcpy(rp32.data(), op.rowptr, sizeof(int) * rp32.size(), cudaMemcpyDeviceToHost));
        std::copy(rp32.begin(), rp32.end(), rp.begin());
    }
    return 0;
}

// stored entries of the sliced layout over these rows: every 32-row slice padded to its longest row
static int64_t sliced_padded_est(const std::vector<int64_t> &rp) {
    const int M = (int)rp.size() - 1;
    int64_t padded = 0;
    for (int s0 = 0; s0 < M; s0 += 32) {
        int64_t mx = 0;
        for (int i = s0; i < std::min(M, s0 + 32); ++i) mx = std::max(mx, rp[i + 1] - rp[i]);
        padded += mx * 32;
    }
    return padded;
}

static void free_sliced(SlicedLayout &s) {
    cudaFree(s.ptr); cudaFree(s.perm); cudaFree(s.col); cudaFree(s.val); cudaFree(s.val32);
    s = SlicedLayout();
}

void sb_free_operator(DevOperator &op) {
    cudaFree(op.rowptr); cudaFree(op.col); cudaFree(op.val); cudaFree(op.blk_row);
    cudaFree(op.brow); cudaFree(op.brow_ptr); cudaFree(op.bcol); cudaFree(op.bval); cudaFree(op.brow_mask);
    cudaFree(op.vIndex); cudaFree(op.send_buf);
    cudaFree(op.hs.epoch); cudaFree(op.hs.tickets); cudaFree(op.hs.segs);
    cudaFree(op.hs.wait_consumed); cudaFree(op.hs.wait_arrived); cudaFree(op.hs.signal_consumed);
    // ghost_buf / x_ext belong to the context's halo arena
    free_sliced(op.sell);
    free_sliced(op.sellp);
    cudaFree(op.sdiag_val);
    cudaFree(op.val32); cudaFree(op.sdiag_val32);
    cudaFree(op.x_round);
    cudaFree(op.rowmid); cudaFree(op.partial);
    op = DevOperator();
}

int sb_upload_operator(saena_b200_ctx *ctx, const saena_b200_operator_desc *d) {
    if (d->level < 0 || d->level > 64) SB_FAIL("upload_operator: level out of range");
    if (d->kind < 0 || d->kind > 2) SB_FAIL("upload_operator: kind must be A, P or R");
    if (d->M < 0 || d->nnz_local < 0 || d->nnz_remote < 0) SB_FAIL("upload_operator: negative size");
    if ((int)ctx->levels.size() <= d->level) ctx->levels.resize(d->level + 1);
    DevLevel &lv = ctx->levels[d->level];
    DevOperator &op = lv.op(d->kind);
    if (ctx->arena) sb_arena_free(ctx);  // ghost areas are re-carved at the next finalize
    if (op.present) sb_free_operator(op);
    op.present = true;
    op.kind = d->kind;
    op.level = d->level;
    op.M = d->M;
    op.int_lo = 0;
    op.int_hi = d->M;
    op.n_local_cols = d->n_local_cols;
    op.col_offset = d->col_offset;
    op.nnz_local = d->nnz_local;
    op.nnz_remote = d->nnz_remote;
    op.use_double = d->use_double != 0;
    op.wide_offsets = d->nnz_local >= (int64_t)INT32_MAX;
    if (d->kind == SAENA_B200_KIND_A) lv.M = d->M;
    const int M = d->M;

    // ---- halo-dominated operator: one CSR over [local | ghost] columns (see DevOperator::merged)
    // Merged when most rows touch ghost columns (deep coarse levels: every row couples to every rank).
    // Also merged when the rows with remote entries are few but SCATTERED: the split path overlaps ONE
    // contiguous run of clean rows with the exchange and sends every other row through the boundary-row
    // kernel (8 or 32 lanes per row, CSR, local + ghost segment) -- right for a slab partition (ghost rows
    // at the two ends of the block), a cliff for transfer operators between a re-split coarse level and
    // the fine level above, or for unstructured matrices: 5 % of scattered rows leave no run worth the
    // name and ~all rows would take the boundary kernel.  (For slab partitions the rows outside the
    // longest clean run ARE the rows with remote entries, and the first rule alone decides, as before.)
    int n_rows_with_remote = 0, n_outside_clean_run = 0;
    for (int64_t k = 0; k < d->nnz_remote; ++k)
        if (d->row_remote[k] < 0 || d->row_remote[k] >= M) SB_FAIL("upload_operator: row_remote out of range");
    if (d->nnz_remote > 0) {
        std::vector<char> has(M, 0);
        for (int64_t k = 0; k < d->nnz_remote; ++k)
            if (!has[d->row_remote[k]]) { has[d->row_remote[k]] = 1; ++n_rows_with_remote; }
        int best = 0;
        for (int i = 0; i < M;) {
            if (has[i]) { ++i; continue; }
            int j = i;
            while (j < M && !has[j]) ++j;
            best = std::max(best, j - i);
            i = j;
        }
        n_outside_clean_run = M - best;
    }
    // (ctx->merge_above, default 0.25, SAENA_B200_MERGE_ABOVE: the fraction of rows with remote entries from which the
    //  split stops paying -- those rows take the boundary-row kernel, the merged operator runs every row on its own
    //  mapping but cannot start before the ghost values are there)
    op.merged = d->nnz_remote > 0 &&
                ((double)n_rows_with_remote >= ctx->merge_above * (double)M ||
                 ((int64_t)n_outside_clean_run * 4 >= M && n_outside_clean_run >= 2 * n_rows_with_remote));
    if (op.merged) {
        const int64_t nl = d->nnz_local, nr = d->nnz_remote, nt = nl + nr;
        std::vector<int64_t> rp(M + 1, 0);
        for (int i = 0; i < M; ++i) rp[i + 1] = d->nnzPerRow_local[i];
        for (int64_t k = 0; k < nr; ++k) ++rp[d->row_remote[k] + 1];
        for (int i = 0; i < M; ++i) rp[i + 1] += rp[i];
        if (rp[M] != nt) SB_FAIL("upload_operator: inconsistent local/remote counts");
        std::vector<int> mc((size_t)nt);
        std::vector<double> mv((size_t)nt);
        std::vector<int64_t> fill(rp.begin(), rp.end() - 1);
        int64_t k = 0;
        for (int i = 0; i < M; ++i)
            for (int j = 0; j < d->nnzPerRow_local[i]; ++j, ++k) {
                const int c = d->col_local[k] - d->col_offset;
                if (c < 0 || c >= d->n_local_cols) SB_FAIL("upload_operator: col_local outside this rank's column block");
                mc[fill[i]] = c;
                mv[fill[i]++] = d->val_local[k];
            }
        k = 0;
        for (int g = 0; g < d->col_remote_size; ++g)
            for (int t = 0; t < d->nnzPerCol_remote[g]; ++t, ++k) {
                const int i = d->row_remote[k];
                mc[fill[i]] = d->n_local_cols + g;
                mv[fill[i]++] = d->val_remote[k];
            }
        if (k != nr) SB_FAIL("upload_operator: sum(nnzPerCol_remote) != nnz_remote");
        op.nnz_local = nt;   // the kernels see one block
        op.nnz_remote = 0;
        op.wide_offsets = nt >= (int64_t)INT32_MAX;
        op.sell_padded_est = sliced_padded_est(rp);
        SB_TRY(upload_rowptr(ctx, op, rp));
        if (!op.wide_offsets) {
            // rows are stored [local columns | ghost columns]: the split point of each row, and the scratch that keeps
            // the local sums across the fused kernel's wait
            std::vector<int> mid((size_t)std::max(M, 1));
            for (int i = 0; i < M; ++i) mid[i] = (int)rp[i] + d->nnzPerRow_local[i];
            SB_TRY(dev_upload(ctx, &op.rowmid, mid.data(), (size_t)M));
            SB_CUDA(cudaMalloc((void **)&op.partial, sizeof(double) * (size_t)std::max(M, 1)));
        }
        SB_TRY(dev_upload(ctx, &op.col, mc.data(), mc.size()));
        SB_TRY(dev_upload(ctx, &op.val, mv.data(), mv.size()));
        // x_ext itself lives in the halo arena (allocated at finalize)
    }

    // ---- local block -> CSR with local column ids
    if (!op.merged) {
        std::vector<int64_t> rp(M + 1, 0);
        for (int i = 0; i < M; ++i) rp[i + 1] = rp[i] + d->nnzPerRow_local[i];
        if (rp[M] != d->nnz_local) SB_FAIL("upload_operator: sum(nnzPerRow_local) != nnz_local");
        op.sell_padded_est = sliced_padded_est(rp);
        SB_TRY(upload_rowptr(ctx, op, rp));
        // columns arrive as GLOBAL ids; make them local on the device and range-check there
        SB_TRY(dev_upload(ctx, &op.col, d->col_local, (size_t)d->nnz_local));
        if (d->nnz_local) {
            int *d_bad = nullptr;
            SB_CUDA(cudaMalloc((void **)&d_bad, sizeof(int)));
            SB_CUDA(cudaMemset(d_bad, 0, sizeof(int)));
            localise_cols_kernel<<<1184, 256>>>(d->nnz_local, op.col, d->col_offset, d->n_local_cols, d_bad);
            int bad = 0;
            SB_CUDA(cudaMemcpy(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost));
            cudaFree(d_bad);
            if (bad) SB_FAIL("upload_operator: col_local outside this rank's column block");
        }
        SB_TRY(dev_upload(ctx, &op.val, d->val_local, (size_t)d->nnz_local));

        // row blocks of the streaming kernel (LPR is fixed later; blocks are cut for the largest
        // row count a CTA can take, STREAM_THREADS, and re-cut in sb_choose_mapping if LPR > 1)
    }

    // ---- remote block: column-major by sender -> row-major over boundary rows
    op.recvSize = d->col_remote_size;
    if (d->nnz_remote > 0 && !op.merged) {
        const int64_t nr = d->nnz_remote;
        std::vector<int> ghost_of((size_t)nr);
        {
            int64_t k = 0;
            for (int j = 0; j < d->col_remote_size; ++j)
                for (int t = 0; t < d->nnzPerCol_remote[j]; ++t) ghost_of[k++] = j;
            if (k != nr) SB_FAIL("upload_operator: sum(nnzPerCol_remote) != nnz_remote");
        }
        std::vector<int> cnt(M + 1, 0);
        for (int64_t k = 0; k < nr; ++k) {
            if (d->row_remote[k] < 0 || d->row_remote[k] >= M) SB_FAIL("upload_operator: row_remote out of range");
            ++cnt[d->row_remote[k] + 1];
        }
        // longest run of rows without remote entries -> interior range, trimmed to multiples of 32
        int best_lo = 0, best_hi = 0;
        for (int i = 0; i < M;) {
            if (cnt[i + 1]) { ++i; continue; }
            int j = i;
            while (j < M && !cnt[j + 1]) ++j;
            if (j - i > best_hi - best_lo) { best_lo = i; best_hi = j; }
            i = j;
        }
        op.int_lo = (best_lo + 31) / 32 * 32;
        op.int_hi = best_hi == M ? M : best_hi / 32 * 32;
        if (op.int_hi < op.int_lo) op.int_hi = op.int_lo;
        std::vector<int> brow, brow_ptr(1, 0);
        std::vector<int> pos(M, -1);
        for (int i = 0; i < M; ++i)
            if (i < op.int_lo || i >= op.int_hi) {   // may hold rows without remote entries: fine
                pos[i] = (int)brow.size();
                brow.push_back(i);
                brow_ptr.push_back(brow_ptr.back() + cnt[i + 1]);
            }
        std::vector<int> fill(brow_ptr.begin(), brow_ptr.end() - 1);
        std::vector<int> bcol((size_t)nr);
        std::vector<double> bval((size_t)nr);
        for (int64_t k = 0; k < nr; ++k) {  // stable: ghost index ascending inside a row
            const int b = pos[d->row_remote[k]];
            bcol[fill[b]] = ghost_of[k];
            bval[fill[b]] = d->val_remote[k];
            ++fill[b];
        }
        std::vector<uint32_t> mask((size_t)(M + 31) / 32, 0u);   // used by the streaming kernel only
        for (int r : brow) mask[r >> 5] |= 1u << (r & 31);
        op.n_brows = (int)brow.size();
        SB_TRY(dev_upload(ctx, &op.brow, brow.data(), brow.size()));
        SB_TRY(dev_upload(ctx, &op.brow_ptr, brow_ptr.data(), brow_ptr.size()));
        SB_TRY(dev_upload(ctx, &op.bcol, bcol.data(), bcol.size()));
        SB_TRY(dev_upload(ctx, &op.bval, bval.data(), bval.size()));
        SB_TRY(dev_upload(ctx, &op.brow_mask, mask.data(), mask.size()));
    }

    // ---- halo plan
    op.vIndexSize = d->vIndexSize;
    if (d->vIndexSize > 0) {
        for (int i = 0; i < d->vIndexSize; ++i)
            if (d->vIndex[i] < 0 || d->vIndex[i] >= d->n_local_cols) SB_FAIL("upload_operator: vIndex out of range");
        SB_TRY(dev_upload(ctx, &op.vIndex, d->vIndex, (size_t)d->vIndexSize));
    }
    const size_t esz = op.use_double ? sizeof(double) : sizeof(float);
    if (op.vIndexSize) SB_CUDA(cudaMalloc(&op.send_buf, (size_t)op.vIndexSize * esz));
    // ghost_buf / x_ext are carved out of the halo arena at finalize (sb_arena_build)
    for (int i = 0; i < d->numSendProc; ++i) {
        const int p = d->sendProcRank[i];
        if (p < 0 || p >= ctx->nranks) SB_FAIL("upload_operator: sendProcRank out of range");
        op.sends.push_back({p, d->vdispls[p], d->sendProcCount[i]});
    }
    for (int i = 0; i < d->numRecvProc; ++i) {
        const int p = d->recvProcRank[i];
        if (p < 0 || p >= ctx->nranks) SB_FAIL("upload_operator: recvProcRank out of range");
        op.recvs.push_back({p, d->rdispls[p], d->recvProcCount[i]});
    }
    if ((!op.sends.empty() || !op.recvs.empty()) && ctx->nranks == 1)
        SB_FAIL("upload_operator: halo plan given but the context has one rank");
    ctx->finalized = false;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// Band operator generated on the device (measurement input, one rank): the pattern and values of
// saena::band_matrix (/root/reference/src/aux_functions2.cpp:1296-1381; experiments/banded.cpp,
// BASELINE.json configs[3]) -- row i holds columns [i-b, i+b] inside [0, n), value 1/(i+j+1).
// 50 M rows x 129 entries are 77 GB: they cannot come through a host upload in a bench run, and
// need 64-bit row offsets.  Same CSR arrays as sb_upload_operator produces from host data
// (tests/test_gpu_parity.py compares the two bit for bit at small n).
// ---------------------------------------------------------------------------------------------
__host__ __device__ static inline long long band_row_start(long long i, long long n, long long b) {
    // entries in rows < i: i full rows minus what the two matrix edges clip
    const long long m = i < b ? i : b;                             // rows clipped on the left
    const long long k = i > n - b ? i - (n - b) : 0;               // rows clipped on the right
    return i * (2 * b + 1) - (m * b - m * (m - 1) / 2) - k * (k + 1) / 2;
}

template <typename OffT>
__global__ void band_fill_kernel(long long n, long long b, OffT *__restrict__ rowptr, int *__restrict__ col,
                                 double *__restrict__ val) {
    const int lane = threadIdx.x & 31;
    const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long i = warp; i < n; i += nwarps) {
        const long long start = band_row_start(i, n, b);
        const long long j0 = i - b < 0 ? 0 : i - b, j1 = i + b > n - 1 ? n - 1 : i + b;
        if (lane == 0) {
            rowptr[i] = (OffT)start;
            if (i == n - 1) rowptr[n] = (OffT)(start + (j1 - j0 + 1));
        }
        for (long long j = j0 + lane; j <= j1; j += 32) {
            col[start + (j - j0)] = (int)j;
            val[start + (j - j0)] = 1.0 / (double)(i + j + 1);
        }
    }
}

int sb_upload_band_operator(saena_b200_ctx *ctx, int level, int n, int half_bandwidth, int sliced_only) {
    if (ctx->nranks != 1) SB_FAIL("upload_band_operator: one rank only (a measurement input)");
    if (level < 0 || level > 64 || n < 1 || half_bandwidth < 0 || half_bandwidth >= n)
        SB_FAIL("upload_band_operator: need 0 <= half_bandwidth < n");
    if ((int)ctx->levels.size() <= level) ctx->levels.resize(level + 1);
    DevLevel &lv = ctx->levels[level];
    DevOperator &op = lv.A;
    if (ctx->arena) sb_arena_free(ctx);
    if (op.present) sb_free_operator(op);
    const long long nn = n, b = half_bandwidth;
    const long long nnz = band_row_start(nn, nn, b);
    op.present = true;
    op.kind = SAENA_B200_KIND_A;
    op.level = level;
    op.M = n;
    op.int_lo = 0;
    op.int_hi = n;
    op.n_local_cols = n;
    op.col_offset = 0;
    op.nnz_local = nnz;
    op.nnz_remote = 0;
    op.use_double = true;
    op.wide_offsets = nnz >= (int64_t)INT32_MAX;
    // slices of 32 consecutive rows differ in length only at the two matrix edges
    op.sell_padded_est = nnz + 32 * 2 * b;
    op.sell_only = sliced_only != 0;
    lv.M = n;
    SB_CUDA(cudaMalloc(&op.rowptr, (op.wide_offsets ? sizeof(int64_t) : sizeof(int)) * ((size_t)n + 1)));
    SB_CUDA(cudaMalloc((void **)&op.col, sizeof(int) * (size_t)nnz));
    SB_CUDA(cudaMalloc((void **)&op.val, sizeof(double) * (size_t)nnz));
    const int blocks = 8 * ctx->sm_count;
    if (op.wide_offsets)
        band_fill_kernel<int64_t><<<blocks, 256, 0, ctx->stream>>>(nn, b, (int64_t *)op.rowptr, op.col, op.val);
    else
        band_fill_kernel<int><<<blocks, 256, 0, ctx->stream>>>(nn, b, (int *)op.rowptr, op.col, op.val);
    SB_CUDA(cudaGetLastError());
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->finalized = false;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// mapping heuristic: lanes per row from nnz/row; short rows stream.  (north_star: "warp-per-row
// or row-block mapping chosen per level by nnz/row".)  Measured crossovers are in DESIGN.md.
// ---------------------------------------------------------------------------------------------
// the largest power of two <= v, at least 1 and at most cap
static int pow2_at_most(double v, int cap) {
    int p = 1;
    while (p * 2 <= v && p < cap) p *= 2;
    return p;
}

void sb_choose_mapping(saena_b200_ctx *ctx, DevOperator &op) {
    const double avg = op.M ? double(op.nnz_local) / op.M : 0.0;
    int m = op.sell_only ? SB_MAPPING_SELL : op.forced_mapping;
    // the sorted sliced layout permutes rows inside 256-row windows: no interior / boundary row ranges, so only for
    // operators without a halo (one rank, or a block that happens to have no remote part)
    if (m == SB_MAPPING_SELLP && (!op.sends.empty() || !op.recvs.empty() || op.merged || op.nnz_remote > 0)) m = 0;
    // the symmetric diagonals only where sb_prepare_operator found the operator eligible
    if (m == SB_MAPPING_SYMDIAG && op.sdiag_n <= 0) m = 0;
    if (m == 0) {
        // short and regular rows: sliced layout (padding <= 15 %); otherwise a sub-warp per row
        // with ~4+ elements per lane.  Crossovers measured on B200, see DESIGN.md.
        // measured on B200 (profiles/r01_mapping_sweep.md): the sliced layout wins whenever its
        // padding is small (7-pt Poisson 5.9 TB/s vs 5.6 best sub-warp; band 61/row 6.8 vs 5.3)
        // ... provided one lane per row still fills the chip: >= ~2 resident threads per lane slot
        // (the 5 416-row x 4 342-nnz level 5 of the 256^3 hierarchy ran at 0.23 TB/s sliced,
        //  profiles/r01_bench_levels.md)
        const bool regular = op.nnz_local > 0 && double(op.sell_padded_est) <= 1.20 * double(op.nnz_local);
        const bool enough_rows = op.M >= 2 * 2048 * ctx->sm_count / 4;  // 151 552 rows on B200
        // an eligible symmetric operator streams its stored diagonals (<= 0.75 of the sliced layout's bytes) instead;
        // the rule takes it where it was measured, up to 4 stored diagonals (the 7-point stencil, 40 registers).  More
        // diagonals (74-78 / 128 registers at 8 / 16) only through set_mapping or the mapping walk, which times them
        if (op.sdiag_n > 0 && op.sdiag.nd <= SYMDIAG_RULE_MAX && enough_rows) m = SB_MAPPING_SYMDIAG;
        else if (regular && enough_rows) m = SB_MAPPING_SELL;
        else {
            // ~4+ elements per lane; rows of hundreds..thousands of entries get 32..256 threads
            m = pow2_at_most((avg + 1.0) / 4.0, 256);
            // few rows: the sub-warp mapping walks its 32 rows in `lanes` dependent steps (2 rows at a
            // time at 16 lanes), and with fewer than ~32 warps per SM nothing hides that chain --
            // measured on the unstructured 2-D hierarchy (profiles/r01_unstructured.md): levels of
            // 715 .. 78 839 rows x ~100 entries all took 57 us per application at 16 lanes/row,
            // 10-18 us with a warp per row, which has no such chain.  (Same row count below which
            // the sliced layout is not chosen: one lane per row cannot fill the chip either.)
            if (m < 32 && op.M <= 32 * 32 * ctx->sm_count) m = 32;
        }
    }
    // the one place a code is made canonical: threads per row 1..256 and streaming lanes 1..32, powers of two
    if (m == SB_MAPPING_SELL || m == SB_MAPPING_SELLP || m == SB_MAPPING_SYMDIAG) op.mapping = m;
    else if (m < 0) op.mapping = -pow2_at_most(-m, 32);
    else op.mapping = pow2_at_most(m, 256);
}

// rows [blk_row[b], blk_row[b+1]) : at most `rows_per_block` rows and STREAM_TILE nnz
static int build_row_blocks(saena_b200_ctx *ctx, DevOperator &op, int rows_per_block) {
    std::vector<int64_t> rp;
    SB_TRY(read_rowptr(ctx, op, rp));
    std::vector<int> blk(1, 0);
    int r = 0;
    while (r < op.M) {
        int e = r;
        const int64_t base = rp[r];
        while (e < op.M && e - r < rows_per_block && rp[e + 1] - base <= STREAM_TILE) ++e;
        if (e == r) e = r + 1;  // one row longer than the tile: alone in its block
        blk.push_back(e);
        r = e;
    }
    cudaFree(op.blk_row);
    op.blk_row = nullptr;
    op.n_blk = (int)blk.size() - 1;
    SB_TRY(dev_upload(ctx, &op.blk_row, blk.data(), blk.size()));
    return 0;
}

// ---------------------------------------------------------------------------------------------
// sliced layouts, built on the device from the CSR arrays (one-time, at finalize):
// 32-slot slices, column-major inside a slice, padded to the slice's longest row
// ---------------------------------------------------------------------------------------------
template <typename OffT>
__global__ void sell_slice_len_kernel(int M, const OffT *__restrict__ rowptr, int *__restrict__ slice_len) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    int len = row < M ? (int)(rowptr[row + 1] - rowptr[row]) : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) len = max(len, __shfl_xor_sync(0xffffffffu, len, o));
    if ((threadIdx.x & 31) == 0 && (row >> 5) < (M + 31) / 32) slice_len[row >> 5] = len;
}

// slot -> row through perm (sorted layout) or slot = row; a slot past the last row holds padding only
template <typename OffT>
__global__ void sliced_fill_kernel(int n_slots, int M, const int *__restrict__ perm, const OffT *__restrict__ rowptr,
                                   const int *__restrict__ col, const double *__restrict__ val,
                                   const long long *__restrict__ slice_ptr, int *__restrict__ scol,
                                   double *__restrict__ sval) {
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= n_slots) return;
    const int slice = slot >> 5, lane = slot & 31;
    const long long base = slice_ptr[slice];
    const int len = (int)((slice_ptr[slice + 1] - base) >> 5);
    const int row = perm ? perm[slot] : (slot < M ? slot : -1);
    OffT a = 0, b = 0;
    if (row >= 0) { a = rowptr[row]; b = rowptr[row + 1]; }
    const int pad_col = (b > a) ? col[b - 1] : 0;  // padding: val 0.0, a column the row already touches
    for (int j = 0; j < len; ++j) {
        const long long dst = base + (long long)j * 32 + lane;
        if (a + j < b) {
            scol[dst] = col[a + j];
            sval[dst] = val[a + j];
        } else {
            scol[dst] = pad_col;
            sval[dst] = 0.0;
        }
    }
}

constexpr int SELLP_WINDOW = 256;  // = the CTA size of spmv_sellp_kernel (mapping 101, below)

// The entries of an existing layout from the operator's CSR arrays: at build time, and again when the values change
// on the same pattern (saena_b200_update_values).  One slot per row, rounded up to whole slices (32 rows) in row
// order, to whole SELLP_WINDOW-row windows over a permutation.
int sb_fill_sliced(saena_b200_ctx *ctx, const DevOperator &op, SlicedLayout &s) {
    const int n_slots = s.perm ? (op.M + SELLP_WINDOW - 1) / SELLP_WINDOW * SELLP_WINDOW : (op.M + 31) / 32 * 32;
    if (n_slots) {
        const int blocks = (n_slots + 255) / 256;
        if (op.wide_offsets)
            sliced_fill_kernel<int64_t><<<blocks, 256, 0, ctx->stream>>>(n_slots, op.M, s.perm, (const int64_t *)op.rowptr,
                                                                         op.col, op.val, s.ptr, s.col, s.val);
        else
            sliced_fill_kernel<int><<<blocks, 256, 0, ctx->stream>>>(n_slots, op.M, s.perm, (const int *)op.rowptr,
                                                                     op.col, op.val, s.ptr, s.col, s.val);
    }
    SB_CUDA(cudaGetLastError());
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// allocates s and fills it from the operator's CSR arrays: sp = element offsets of the 32-slot slices, perm = slot ->
// row or nullptr
static int build_sliced(saena_b200_ctx *ctx, DevOperator &op, SlicedLayout &s, const std::vector<long long> &sp,
                        const std::vector<int> *perm) {
    const int64_t padded = sp.back();
    SB_TRY(dev_upload(ctx, &s.ptr, sp.data(), sp.size()));
    if (perm) SB_TRY(dev_upload(ctx, &s.perm, perm->data(), perm->size()));
    SB_CUDA(cudaMalloc((void **)&s.col, sizeof(int) * std::max<int64_t>(padded, 1)));
    SB_CUDA(cudaMalloc((void **)&s.val, sizeof(double) * std::max<int64_t>(padded, 1)));
    return sb_fill_sliced(ctx, op, s);
}

// the slice lengths come from the row offsets on the device: the row offsets of a device-generated band operator
// (50 M rows) are never read back
static int build_sell(saena_b200_ctx *ctx, DevOperator &op) {
    if (op.sell.ptr) return 0;
    const int M = op.M;
    const int ns = (M + 31) / 32;
    int *d_len = nullptr;
    SB_CUDA(cudaMalloc((void **)&d_len, sizeof(int) * std::max(ns, 1)));
    const int blocks = (ns * 32 + 255) / 256;
    if (ns) {
        if (op.wide_offsets)
            sell_slice_len_kernel<int64_t><<<blocks, 256, 0, ctx->stream>>>(M, (const int64_t *)op.rowptr, d_len);
        else
            sell_slice_len_kernel<int><<<blocks, 256, 0, ctx->stream>>>(M, (const int *)op.rowptr, d_len);
    }
    std::vector<int> len(ns);
    SB_CUDA(cudaMemcpyAsync(len.data(), d_len, sizeof(int) * ns, cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    cudaFree(d_len);
    std::vector<long long> sp(ns + 1, 0);
    for (int s0 = 0; s0 < ns; ++s0) sp[s0 + 1] = sp[s0] + (long long)len[s0] * 32;
    SB_TRY(build_sliced(ctx, op, op.sell, sp, nullptr));
    if (op.sell_only) {
        // the sliced copy is the operator from here on: give the CSR entries back (half the footprint)
        cudaFree(op.col);
        cudaFree(op.val);
        op.col = nullptr;
        op.val = nullptr;
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------
// sorted sliced layout (mapping 101): rows sorted by length, longest first, inside windows of SELLP_WINDOW
// consecutive rows; the permutation is made on the host from the row offsets, the entries are moved on the device
// ---------------------------------------------------------------------------------------------
// host only: slot -> row (rows of each SELLP_WINDOW-row window sorted by length, longest first, stable; -1 where the
// last window runs past M) and the element offset of every 32-slot slice (its longest row's length x 32).
// perm[ceil(M / 256) * 256], slice_ptr[ceil(M / 256) * 8 + 1].
void sb_sellp_layout(int M, const int64_t *rp, int *perm, long long *sp) {
    const int n_win = (M + SELLP_WINDOW - 1) / SELLP_WINDOW;
    sp[0] = 0;
    for (int w = 0; w < n_win; ++w) {
        const int r0 = w * SELLP_WINDOW, r1 = std::min(M, r0 + SELLP_WINDOW);
        int *p = perm + (size_t)w * SELLP_WINDOW;
        for (int k = 0; k < SELLP_WINDOW; ++k) p[k] = r0 + k < r1 ? r0 + k : -1;
        std::stable_sort(p, p + (r1 - r0), [&](int x, int y) { return rp[x + 1] - rp[x] > rp[y + 1] - rp[y]; });
        for (int k = 0; k < SELLP_WINDOW / 32; ++k) {
            const int first = p[k * 32];                        // the longest row of the slice (or none: -1)
            const long long len = first >= 0 ? (long long)(rp[first + 1] - rp[first]) : 0;
            const int sl = w * (SELLP_WINDOW / 32) + k;
            sp[sl + 1] = sp[sl] + len * 32;
        }
    }
}

static int build_sellp(saena_b200_ctx *ctx, DevOperator &op) {
    if (op.sellp.ptr) return 0;
    if (!op.col || !op.val) SB_FAIL("sorted sliced layout: the CSR entries of this operator were released");
    const int n_slots = (op.M + SELLP_WINDOW - 1) / SELLP_WINDOW * SELLP_WINDOW;
    std::vector<int64_t> rp;
    SB_TRY(read_rowptr(ctx, op, rp));
    std::vector<int> perm((size_t)std::max(n_slots, 1), -1);
    std::vector<long long> sp((size_t)n_slots / 32 + 1, 0);
    sb_sellp_layout(op.M, rp.data(), perm.data(), sp.data());
    return build_sliced(ctx, op, op.sellp, sp, &perm);
}

// ---------------------------------------------------------------------------------------------
// symmetric diagonals (mapping 103): eligibility from the distinct offsets col - row (one device pass, bounded table)
// and a host rule; the diagonals filled from the CSR and checked for exact symmetry on the device
// ---------------------------------------------------------------------------------------------
constexpr int SD_TABLE = 32;           // distinct offsets collected before the operator is given up
constexpr int SD_EMPTY = INT_MIN;      // free table slot (no offset of a square operator is INT_MIN)
enum { SD_OVERFLOW = 1, SD_UNSORTED = 2, SD_ASYMMETRIC = 4 };

// offset -> its slot in the table (inserted if new); false when the table is full
__device__ __forceinline__ bool sd_insert(int *t, int off) {
    for (int j = 0; j < SD_TABLE; ++j) {
        int v = *(volatile int *)(t + j);
        if (v == SD_EMPTY) v = atomicCAS(t + j, SD_EMPTY, off);
        if (v == SD_EMPTY || v == off) return true;
    }
    return false;
}

// the distinct offsets of the operator into table[SD_TABLE] (per CTA in shared memory, then merged); flags: more than
// SD_TABLE offsets, or a row whose columns do not strictly ascend (the kernel's sum order is the CSR's column order)
template <typename OffT>
__global__ void sd_offsets_kernel(int M, const OffT *__restrict__ rowptr, const int *__restrict__ col, int *table,
                                  int *flags) {
    __shared__ int s[SD_TABLE];
    if (threadIdx.x < SD_TABLE) s[threadIdx.x] = SD_EMPTY;
    __syncthreads();
    int f = 0;
    for (int row = blockIdx.x * blockDim.x + threadIdx.x; row < M; row += gridDim.x * blockDim.x) {
        // more than SD_TABLE offsets anywhere: the operator is given up, nothing more to scan
        if (*(volatile int *)flags & SD_OVERFLOW) break;
        int prev = INT_MIN;
        for (OffT k = rowptr[row]; k < rowptr[row + 1]; ++k) {
            const int c = col[k];
            if (c <= prev) f |= SD_UNSORTED;
            prev = c;
            if (!sd_insert(s, c - row)) {
                atomicOr(flags, SD_OVERFLOW);
                break;
            }
        }
    }
    if (f) atomicOr(flags, f);
    __syncthreads();
    if (threadIdx.x < SD_TABLE && s[threadIdx.x] != SD_EMPTY && !sd_insert(table, s[threadIdx.x])) atomicOr(flags, SD_OVERFLOW);
}

__device__ __forceinline__ int sd_index(const SymDiagOffsets &s, int k) {
    for (int q = 0; q < s.nd; ++q)
        if (s.off[q] == k) return q;
    return -1;
}

// upper entries (col >= row) into d_q[row]: each slot written once (columns strictly ascend)
template <typename OffT>
__global__ void sd_fill_kernel(int M, const OffT *__restrict__ rowptr, const int *__restrict__ col,
                               const double *__restrict__ val, const SymDiagOffsets s, double *__restrict__ d,
                               int *flags) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= M) return;
    for (OffT k = rowptr[row]; k < rowptr[row + 1]; ++k) {
        const int c = col[k];
        if (c < row) continue;
        const int q = sd_index(s, c - row);
        if (q < 0) { atomicOr(flags, SD_ASYMMETRIC); continue; }
        d[(size_t)q * (size_t)M + row] = val[k];
    }
}

// every lower entry a_{row,c} (c < row): row c holds column `row`, and a_{row,c} has the bits of d_{row-c}[c] (that
// entry); balance += lower - upper off-diagonal entries, 0 when the pattern is symmetric
template <typename OffT>
__global__ void sd_check_kernel(int M, const OffT *__restrict__ rowptr, const int *__restrict__ col,
                                const double *__restrict__ val, const SymDiagOffsets s, const double *__restrict__ d,
                                int *flags, unsigned long long *balance) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    long long bal = 0;
    bool bad = false;
    if (row < M) {
        for (OffT k = rowptr[row]; k < rowptr[row + 1]; ++k) {
            const int c = col[k];
            if (c > row) --bal;
            if (c >= row) continue;
            ++bal;
            const int q = sd_index(s, row - c);
            OffT lo = rowptr[c], hi = rowptr[c + 1];   // row c's columns ascend: binary search for `row`
            while (lo < hi) {
                const OffT mid = lo + (hi - lo) / 2;
                if (col[mid] < row) lo = mid + 1; else hi = mid;
            }
            if (q < 0 || lo == rowptr[c + 1] || col[lo] != row ||
                __double_as_longlong(val[k]) != __double_as_longlong(d[(size_t)q * (size_t)M + c]))
                bad = true;
        }
    }
    if (bad) atomicOr(flags, SD_ASYMMETRIC);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) bal += __shfl_xor_sync(0xffffffffu, bal, o);
    if ((threadIdx.x & 31) == 0 && bal) atomicAdd(balance, (unsigned long long)bal);
}

int sb_symdiag_plan(int M, int n_offsets, const int *offsets, int64_t nnz, int64_t padded_est, int *stored) {
    if (M <= 0 || nnz <= 0 || n_offsets < 0 || n_offsets > SD_TABLE) return 0;
    std::vector<int> off(offsets, offsets + n_offsets);
    std::sort(off.begin(), off.end());
    off.erase(std::unique(off.begin(), off.end()), off.end());
    std::vector<int> pos;
    for (int k : off) {
        if (k <= -M || k >= M) return 0;
        if (!std::binary_search(off.begin(), off.end(), -k)) return 0;   // every offset has its mirror
        if (k > 0) pos.push_back(k);
    }
    const int nd = 1 + (int)pos.size();
    if (nd > SYMDIAG_MAX) return 0;
    // clearly fewer bytes than the sliced layout: values of the stored diagonals against values + column ids
    if (8.0 * nd * (double)M > 0.75 * 12.0 * (double)padded_est) return 0;
    stored[0] = 0;
    std::copy(pos.begin(), pos.end(), stored + 1);
    return nd;
}

// one rank, no halo, square, CSR entries kept
static bool symdiag_candidate(const saena_b200_ctx *ctx, const DevOperator &op) {
    return ctx->nranks == 1 && !op.merged && !op.sell_only && op.nnz_remote == 0 && op.sends.empty() &&
           op.recvs.empty() && op.M > 0 && op.M == op.n_local_cols && op.nnz_local > 0 && op.col && op.val;
}

// op.sdiag_n from the operator's offsets and the host rule (pattern only; the values are checked at every fill)
static int probe_symdiag(saena_b200_ctx *ctx, DevOperator &op) {
    cudaFree(op.sdiag_val);   // filled from values that may have changed since
    op.sdiag_val = nullptr;
    op.sdiag_n = 0;
    if (!symdiag_candidate(ctx, op)) return 0;
    int *dev = nullptr;   // [SD_TABLE] offsets, [1] flags
    SB_CUDA(cudaMalloc((void **)&dev, sizeof(int) * (SD_TABLE + 1)));
    std::vector<int> h(SD_TABLE + 1, SD_EMPTY);
    h[SD_TABLE] = 0;
    SB_CUDA(cudaMemcpyAsync(dev, h.data(), sizeof(int) * h.size(), cudaMemcpyHostToDevice, ctx->stream));
    const int blocks = std::min((op.M + 255) / 256, 8 * ctx->sm_count);
    if (op.wide_offsets)
        sd_offsets_kernel<int64_t><<<blocks, 256, 0, ctx->stream>>>(op.M, (const int64_t *)op.rowptr, op.col, dev, dev + SD_TABLE);
    else
        sd_offsets_kernel<int><<<blocks, 256, 0, ctx->stream>>>(op.M, (const int *)op.rowptr, op.col, dev, dev + SD_TABLE);
    SB_CUDA(cudaGetLastError());
    SB_CUDA(cudaMemcpyAsync(h.data(), dev, sizeof(int) * h.size(), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    cudaFree(dev);
    if (h[SD_TABLE]) return 0;
    std::vector<int> off;
    for (int j = 0; j < SD_TABLE; ++j)
        if (h[j] != SD_EMPTY) off.push_back(h[j]);
    SymDiagOffsets s;
    s.nd = sb_symdiag_plan(op.M, (int)off.size(), off.data(), op.nnz_local, op.sell_padded_est, s.off);
    op.sdiag = s;
    op.sdiag_n = s.nd;
    return 0;
}

// The diagonals from the operator's CSR arrays, then the symmetry check: at build time, and again when the values
// change on the same pattern (saena_b200_update_values).  *symmetric false: the values are not exactly symmetric.
static int fill_symdiag(saena_b200_ctx *ctx, DevOperator &op, bool *symmetric) {
    const int M = op.M, blocks = (M + 255) / 256;
    const SymDiagOffsets &s = op.sdiag;
    int *flags = nullptr;   // [0] flags, then (8-byte aligned) the balance
    SB_CUDA(cudaMalloc((void **)&flags, 2 * sizeof(unsigned long long)));
    unsigned long long *balance = (unsigned long long *)flags + 1;
    SB_CUDA(cudaMemsetAsync(flags, 0, 2 * sizeof(unsigned long long), ctx->stream));
    SB_CUDA(cudaMemsetAsync(op.sdiag_val, 0, sizeof(double) * (size_t)s.nd * (size_t)M, ctx->stream));
    if (op.wide_offsets) {
        const int64_t *rp = (const int64_t *)op.rowptr;
        sd_fill_kernel<int64_t><<<blocks, 256, 0, ctx->stream>>>(M, rp, op.col, op.val, s, op.sdiag_val, flags);
        sd_check_kernel<int64_t><<<blocks, 256, 0, ctx->stream>>>(M, rp, op.col, op.val, s, op.sdiag_val, flags, balance);
    } else {
        const int *rp = (const int *)op.rowptr;
        sd_fill_kernel<int><<<blocks, 256, 0, ctx->stream>>>(M, rp, op.col, op.val, s, op.sdiag_val, flags);
        sd_check_kernel<int><<<blocks, 256, 0, ctx->stream>>>(M, rp, op.col, op.val, s, op.sdiag_val, flags, balance);
    }
    SB_CUDA(cudaGetLastError());
    unsigned long long h[2] = {0ull, 0ull};   // the int flags are the low half of h[0]
    SB_CUDA(cudaMemcpyAsync(h, flags, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    cudaFree(flags);
    *symmetric = h[0] == 0ull && h[1] == 0ull;
    return 0;
}

// allocates and fills the diagonals; an operator whose values are not symmetric loses its eligibility (freed)
static int build_symdiag(saena_b200_ctx *ctx, DevOperator &op, bool *ok) {
    *ok = true;
    if (op.sdiag_val) return 0;
    SB_CUDA(cudaMalloc((void **)&op.sdiag_val, sizeof(double) * (size_t)op.sdiag.nd * (size_t)op.M));
    SB_TRY(fill_symdiag(ctx, op, ok));
    if (!*ok) {
        cudaFree(op.sdiag_val);
        op.sdiag_val = nullptr;
        op.sdiag_n = 0;
    }
    return 0;
}

int sb_refresh_symdiag(saena_b200_ctx *ctx, DevOperator &op) {
    if (op.mapping != SB_MAPPING_SYMDIAG) {
        op.sdiag_n = -1;   // probed again (and a stale copy freed) the next time the operator is prepared
        return 0;
    }
    bool ok = false;
    SB_TRY(fill_symdiag(ctx, op, &ok));
    if (ok) return 0;
    cudaFree(op.sdiag_val);
    op.sdiag_val = nullptr;
    op.sdiag_n = 0;
    op.forced_mapping = SB_MAPPING_SELL;
    return sb_prepare_operator(ctx, op);
}

// copies of the entries in layouts the operator no longer uses (a mapping walk builds them to time them)
void sb_drop_unused_layouts(DevOperator &op) {
    if (op.mapping != SB_MAPPING_SELLP) free_sliced(op.sellp);
    if (op.mapping != SB_MAPPING_SELL && !op.sell_only) free_sliced(op.sell);
    if (op.mapping != SB_MAPPING_SYMDIAG) {
        cudaFree(op.sdiag_val);
        op.sdiag_val = nullptr;
    }
}

int sb_prepare_operator(saena_b200_ctx *ctx, DevOperator &op) {
    if (!op.present) return 0;
    if (op.sdiag_n < 0) SB_TRY(probe_symdiag(ctx, op));
    sb_choose_mapping(ctx, op);
    if (op.mapping == SB_MAPPING_SYMDIAG) {
        bool ok = false;
        SB_TRY(build_symdiag(ctx, op, &ok));
        if (!ok) sb_choose_mapping(ctx, op);   // not symmetric after all: the rule's choice (or the forced one)
    }
    if (op.mapping < 0) SB_TRY(build_row_blocks(ctx, op, STREAM_THREADS / -op.mapping));
    if (op.mapping == SB_MAPPING_SELL) SB_TRY(build_sell(ctx, op));
    if (op.mapping == SB_MAPPING_SELLP) SB_TRY(build_sellp(ctx, op));
    return 0;
}

// ---------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------
template <int EPI, typename OffT>
static int launch_local(saena_b200_ctx *ctx, DevOperator &op, const double *x, const EpiArgs &e) {
    const OffT *rp = (const OffT *)op.rowptr;
    cudaStream_t s = ctx->stream;
    const bool stream = op.mapping < 0;
    // rows [lo, hi): everything when there is no halo, else the interior range
    const int lo = stream ? 0 : op.int_lo, hi = stream ? op.M : op.int_hi;
    const int nrows = hi - lo;
    if (nrows <= 0) return 0;
    ++ctx->launches;
    if (op.mapping == SB_MAPPING_SYMDIAG) {
        // whole operator (no halo): one thread per row
        const int blocks = (op.M + 255) / 256;
        const double *d = op.sdiag_val;
        if (op.sdiag.nd <= 4) spmv_symdiag_kernel<4, EPI><<<blocks, 256, 0, s>>>(op.M, d, op.sdiag, x, e);
        else if (op.sdiag.nd <= 8) spmv_symdiag_kernel<8, EPI><<<blocks, 256, 0, s>>>(op.M, d, op.sdiag, x, e);
        else spmv_symdiag_kernel<SYMDIAG_MAX, EPI><<<blocks, 256, 0, s>>>(op.M, d, op.sdiag, x, e);
        return 0;
    }
    if (op.mapping == SB_MAPPING_SELLP) {
        // whole operator (no halo, see sb_choose_mapping): one CTA per 256-row window
        spmv_sellp_kernel<EPI><<<(op.M + 255) / 256, 256, 0, s>>>(op.M, op.sellp.ptr, op.sellp.perm, op.sellp.col,
                                                                   op.sellp.val, x, e);
        return 0;
    }
    if (stream) {
        switch (-op.mapping) {
#define SB_STREAM_CASE(L)                                                                          \
    case L:                                                                                        \
        spmv_stream_kernel<L, EPI, OffT><<<op.n_blk, STREAM_THREADS, 0, s>>>(                      \
            op.M, rp, op.col, op.val, x, e, op.brow_mask, op.blk_row);                             \
        break;
            SB_STREAM_CASE(1) SB_STREAM_CASE(2) SB_STREAM_CASE(4) SB_STREAM_CASE(8)
            SB_STREAM_CASE(16) SB_STREAM_CASE(32)
#undef SB_STREAM_CASE
        }
        return 0;
    }
    const int blocks = sb_mapping_blocks(op.mapping, nrows);
    const bool known = sb_dispatch_mapping(op.mapping, [&](auto map) {
        constexpr int MAP = decltype(map)::value;
        if constexpr (MAP == SB_MAPPING_SELL)
            spmv_sell_kernel<EPI><<<blocks, 256, 0, s>>>(lo, hi, op.sell.ptr, op.sell.col, op.sell.val, x, e, nullptr);
        else if constexpr (MAP >= 32)
            spmv_rowgroup_kernel<MAP, EPI, OffT><<<blocks, 256, 0, s>>>(lo, hi, rp, op.col, op.val, x, e, nullptr);
        else
            spmv_vec_kernel<MAP, EPI, OffT><<<blocks, 256, 0, s>>>(lo, hi, rp, op.col, op.val, x, e, nullptr);
    });
    if (!known) SB_FAIL("apply: unknown mapping");
    return 0;
}

template <int EPI, typename OffT>
static void launch_boundary(saena_b200_ctx *ctx, DevOperator &op, const double *x, const EpiArgs &e) {
    if (op.n_brows == 0) return;
    ++ctx->launches;
    const OffT *rp = (const OffT *)op.rowptr;
    // a warp per boundary row once rows are long (coarse levels, R), 8 lanes for stencil rows
    const bool wide = op.avg_nnz_row() >= 48.0;
    const int threads = 256, rows_per_block = threads / (wide ? 32 : 8);
    const int blocks = (op.n_brows + rows_per_block - 1) / rows_per_block;
#define SB_BND(L, G, GHOST, EPOCH)                                                                 \
    spmv_boundary_kernel<L, EPI, OffT, G><<<blocks, threads, 0, ctx->stream>>>(                    \
        op.n_brows, op.brow, rp, op.col, op.val, op.brow_ptr, op.bcol, op.bval, x,                 \
        (const G *)(GHOST), EPOCH, op.recvSize, e)
    if (op.p2p) {
        // peer-memory exchange: doubles (the sender rounded through float when use_double is false), two buffers
        if (wide) SB_BND(32, double, op.ghost_d, op.hs.epoch); else SB_BND(8, double, op.ghost_d, op.hs.epoch);
    } else if (op.use_double) {
        if (wide) SB_BND(32, double, op.ghost_buf, nullptr); else SB_BND(8, double, op.ghost_buf, nullptr);
    } else {
        if (wide) SB_BND(32, float, op.ghost_buf, nullptr); else SB_BND(8, float, op.ghost_buf, nullptr);
    }
#undef SB_BND
}

// The compute stream joins the comm stream (its own pack / exchange is done: x may be overwritten by the caller, and
// nothing of this application is still waiting for an SM), then waits for the ghost values.
static int wait_halo(saena_b200_ctx *ctx, DevOperator &op) {
    SB_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_halo, 0));
    if (op.p2p) return sb_p2p_wait_arrived(ctx, op, ctx->stream);
    return 0;
}

template <int EPI>
static int apply_epi(saena_b200_ctx *ctx, DevOperator &op, const double *x, const EpiArgs &e) {
    // several ranks, peers imported: exchange + SpMV as one kernel (fused_halo.cu)
    if (sb_fused_eligible(op)) return sb_apply_fused(ctx, op, x, EPI, e);
    const bool has_halo = !op.sends.empty() || !op.recvs.empty();
    const bool halo = has_halo && ctx->apply_mode != 1;
    const bool compute = ctx->apply_mode != 2;
    if (halo && ctx->detached) SB_FAIL("apply: a detached context has no peer to exchange ghost values with");
    if (halo) {
        // pack + exchange on the comm stream, both overlapped with the interior rows: the comm
        // stream only waits for x to be ready (ev_packed marks that point of the compute stream),
        // the compute stream goes straight on to the interior kernel
        SB_CUDA(cudaEventRecord(ctx->ev_packed, ctx->stream));
        SB_CUDA(cudaStreamWaitEvent(ctx->comm_stream, ctx->ev_packed, 0));
        if (op.p2p) {
            // peer-memory path: the pack kernel stores straight into the neighbours' landing areas
            // over NVLink and raises their "arrived" counters; no send buffer, no NCCL rendezvous
            SB_TRY(sb_p2p_pack(ctx, op, x, ctx->comm_stream));
        } else {
            if (op.vIndexSize) {
                ++ctx->launches;
                const int blocks = (op.vIndexSize + 255) / 256;
                if (op.use_double)
                    halo_pack_kernel<double><<<blocks, 256, 0, ctx->comm_stream>>>(op.vIndexSize, op.vIndex, x,
                                                                                   (double *)op.send_buf);
                else
                    halo_pack_kernel<float><<<blocks, 256, 0, ctx->comm_stream>>>(op.vIndexSize, op.vIndex, x,
                                                                                  (float *)op.send_buf);
            }
            SB_TRY(sb_halo_exchange(ctx, op, ctx->comm_stream));
        }
        SB_CUDA(cudaEventRecord(ctx->ev_halo, ctx->comm_stream));
    }
    if (op.merged) {
        // x_ext = [x | ghosts], then one ordinary SpMV over the extended columns
        if (compute && op.n_local_cols)
            SB_CUDA(cudaMemcpyAsync(op.x_ext, x, sizeof(double) * op.n_local_cols, cudaMemcpyDeviceToDevice, ctx->stream));
        if (halo) SB_TRY(wait_halo(ctx, op));
        if (compute) {
            if (op.p2p) {
                SB_TRY(sb_p2p_gather_ghosts(ctx, op, op.x_ext + op.n_local_cols, ctx->stream));
            } else if (!op.use_double && op.recvSize) {
                ++ctx->launches;
                widen_ghost_kernel<<<(op.recvSize + 255) / 256, 256, 0, ctx->stream>>>(
                    op.recvSize, (const float *)op.ghost_buf, op.x_ext + op.n_local_cols);
            }
            if (op.wide_offsets) SB_TRY((launch_local<EPI, int64_t>(ctx, op, op.x_ext, e)));
            else SB_TRY((launch_local<EPI, int>(ctx, op, op.x_ext, e)));
        }
        if (halo && op.p2p) SB_TRY(sb_p2p_release(ctx, op, ctx->stream));
        SB_CUDA(cudaGetLastError());
        return 0;
    }
    if (compute) {
        if (op.wide_offsets) SB_TRY((launch_local<EPI, int64_t>(ctx, op, x, e)));
        else SB_TRY((launch_local<EPI, int>(ctx, op, x, e)));
    }
    if (halo) SB_TRY(wait_halo(ctx, op));
    if (has_halo && compute) {
        if (op.wide_offsets) launch_boundary<EPI, int64_t>(ctx, op, x, e);
        else launch_boundary<EPI, int>(ctx, op, x, e);
    }
    if (halo && op.p2p) SB_TRY(sb_p2p_release(ctx, op, ctx->stream));
    SB_CUDA(cudaGetLastError());
    return 0;
}

// matvec_dense_float (src/saena_matrix_dense.cpp:281-282): v_send_f = float(v) for the whole vector
static __global__ void round_through_float_kernel(int n, const double *__restrict__ in, double *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (double)(float)in[i];
}

int sb_apply(saena_b200_ctx *ctx, DevOperator &op, const double *x, int epi, const EpiArgs &args) {
    if (!op.present) SB_FAIL("apply: operator was not uploaded");
    if (op.use_dense && !op.use_double && op.n_local_cols > 0) {
        // a level the reference applies through saena_matrix_dense with float precision: the operand of
        // the product is float(x) everywhere (the epilogue still reads the unrounded iterate, args.u_in)
        if (!op.x_round) SB_FAIL("apply: dense operator without its rounded-input buffer");
        ++ctx->launches;
        round_through_float_kernel<<<(op.n_local_cols + 255) / 256, 256, 0, ctx->stream>>>(op.n_local_cols, x, op.x_round);
        x = op.x_round;
    }
    switch (epi) {
        case EPI_PLAIN: return apply_epi<EPI_PLAIN>(ctx, op, x, args);
        case EPI_RESIDUAL: return apply_epi<EPI_RESIDUAL>(ctx, op, x, args);
        case EPI_CHEB_FIRST: return apply_epi<EPI_CHEB_FIRST>(ctx, op, x, args);
        case EPI_CHEB_NEXT: return apply_epi<EPI_CHEB_NEXT>(ctx, op, x, args);
        case EPI_JACOBI: return apply_epi<EPI_JACOBI>(ctx, op, x, args);
        case EPI_SUB: return apply_epi<EPI_SUB>(ctx, op, x, args);
    }
    SB_FAIL("apply: unknown epilogue");
}

// algorithmic bytes of w = Op v (SURVEY.md 8d): nnz*(8+4) + M*p (row offsets) + N*8 (x once) + M*8 (w); on the
// symmetric diagonals each stored diagonal once (its second, lagging read is expected from L2) + x + w.  vb = 4: the
// FP32 copy, 4-byte values and vector elements (the column ids and row offsets stay as they are)
int64_t sb_operator_bytes(const DevOperator &op, int vb) {
    if (op.mapping == SB_MAPPING_SYMDIAG) return vb * (int64_t)op.sdiag.nd * op.M + (int64_t)op.n_local_cols * vb + (int64_t)op.M * vb;
    const int64_t p = op.wide_offsets ? 8 : 4;
    return (op.nnz_local + op.nnz_remote) * (vb + 4) + (int64_t)op.M * p + (int64_t)op.n_local_cols * vb +
           (int64_t)op.M * vb;
}
