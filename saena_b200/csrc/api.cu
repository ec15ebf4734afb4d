// api.cu -- the extern "C" entry points declared in include/saena_b200.h.
#include <math.h>
#include <string.h>

#include <algorithm>

#include <stdlib.h>
#include <time.h>

#include "common.h"

thread_local std::string g_sb_init_error;
int sb_prepare_operator(saena_b200_ctx *ctx, DevOperator &op);

extern "C" {

const char *saena_b200_last_error(const saena_b200_ctx *ctx) {
    return ctx ? ctx->error.c_str() : g_sb_init_error.c_str();
}

int saena_b200_nccl_unique_id(void *id_out) { return sb_nccl_unique_id(id_out, g_sb_init_error); }

static int init_body(saena_b200_ctx *ctx, const void *nccl_id) {
    int ndev = 0;
    SB_CUDA(cudaGetDeviceCount(&ndev));
    if (ndev == 0) SB_FAIL("no CUDA device: this library has no CPU path");
    if (ctx->device < 0 || ctx->device >= ndev) SB_FAIL("init: device_id out of range");
    SB_CUDA(cudaSetDevice(ctx->device));
    cudaDeviceProp prop;
    SB_CUDA(cudaGetDeviceProperties(&prop, ctx->device));
    ctx->sm_count = prop.multiProcessorCount;
    // the comm stream carries the pack kernels of the separate-launch halo: highest priority, so that its few CTAs are
    // placed as soon as an SM has room while the interior-row kernel of the same application fills the chip
    int prio_lo = 0, prio_hi = 0;
    SB_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    SB_CUDA(cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_lo));
    SB_CUDA(cudaStreamCreateWithPriority(&ctx->comm_stream, cudaStreamNonBlocking, prio_hi));
    SB_CUDA(cudaEventCreateWithFlags(&ctx->ev_packed, cudaEventDisableTiming));
    SB_CUDA(cudaEventCreateWithFlags(&ctx->ev_halo, cudaEventDisableTiming));
    SB_CUDA(cudaEventCreate(&ctx->ev_t0));
    SB_CUDA(cudaEventCreate(&ctx->ev_t1));
    SB_CUDA(cudaMalloc((void **)&ctx->red_partials, sizeof(double) * RED_MAX_BLOCKS * 4));
    SB_CUDA(cudaMalloc((void **)&ctx->red_counter, sizeof(unsigned int)));
    SB_CUDA(cudaMemset(ctx->red_counter, 0, sizeof(unsigned int)));
    // Krylov scalars followed by the halo fault record: one device-to-host copy per iteration brings both
    static_assert(sizeof(double) == sizeof(unsigned long long), "fault words share the scalar buffer");
    SB_CUDA(cudaMalloc((void **)&ctx->scalars, sizeof(double) * (S_COUNT + S_FAULT_WORDS)));
    SB_CUDA(cudaMemset(ctx->scalars, 0, sizeof(double) * (S_COUNT + S_FAULT_WORDS)));
    SB_CUDA(cudaMallocHost((void **)&ctx->scalars_host, sizeof(double) * (S_COUNT + S_FAULT_WORDS)));
    memset(ctx->scalars_host, 0, sizeof(double) * (S_COUNT + S_FAULT_WORDS));
    ctx->fault_dev = (unsigned long long *)(ctx->scalars + S_COUNT);
    if (!ctx->detached) SB_TRY(sb_nccl_init(ctx, nccl_id));
    return 0;
}

static int init_common(saena_b200_ctx **ctx_out, int device_id, int rank, int nranks, const void *nccl_id, bool detached);

int saena_b200_init(saena_b200_ctx **ctx_out, int device_id, int rank, int nranks, const void *nccl_id) {
    return init_common(ctx_out, device_id, rank, nranks, nccl_id, false);
}

// Profiling aid: one rank's share of an nranks-way partition on ONE GPU, with no peer behind it.
// Nothing that needs a peer works (any exchange fails loudly); what does work is the compute side
// of the distributed kernels on that share -- saena_b200_time_matvec_compute_only -- which is how
// the fused halo kernel's interior / ghost-row roles get under ncu (ncu cannot follow a multi-rank
// command).  Ghost values are whatever the landing areas hold (zeros).
int saena_b200_init_detached(saena_b200_ctx **ctx_out, int device_id, int rank, int nranks) {
    return init_common(ctx_out, device_id, rank, nranks, nullptr, true);
}

static int init_common(saena_b200_ctx **ctx_out, int device_id, int rank, int nranks, const void *nccl_id, bool detached) {
    *ctx_out = nullptr;
    if (nranks < 1 || rank < 0 || rank >= nranks) {
        g_sb_init_error = "init: bad rank / nranks";
        return 1;
    }
    saena_b200_ctx *ctx = new saena_b200_ctx();
    ctx->device = device_id;
    ctx->rank = rank;
    ctx->nranks = nranks;
    ctx->detached = detached;
    if (const char *gm = getenv("SAENA_B200_GRAPH_MULTI")) ctx->use_graphs_multi = atoi(gm) != 0;
    if (const char *hf = getenv("SAENA_B200_HALO_FUSED")) ctx->fused_default = atoi(hf) != 0;
    if (const char *nv = getenv("SAENA_B200_NVTX")) ctx->nvtx = atoi(nv) != 0;
    if (const char *m = getenv("SAENA_B200_MERGE_ABOVE")) ctx->merge_above = atof(m);
    if (const char *m = getenv("SAENA_B200_MERGED_SPLIT")) ctx->merged_split = atoi(m) != 0;
    if (const char *t = getenv("SAENA_B200_HALO_TIMEOUT_MS")) ctx->halo_timeout_ns = (unsigned long long)(atof(t) * 1e6);
    if (const char *t = getenv("SAENA_B200_SYNC_TIMEOUT_S")) ctx->sync_timeout_s = atof(t);
    if (init_body(ctx, nccl_id)) {
        g_sb_init_error = ctx->error;
        delete ctx;
        return 1;
    }
    *ctx_out = ctx;
    return 0;
}

static void free_level_work(DevLevel &lv, bool owns_rhs) {
    cudaFree(lv.u[0]); cudaFree(lv.u[1]); cudaFree(lv.d); cudaFree(lv.res); cudaFree(lv.xfer_old);
    if (owns_rhs) cudaFree(lv.rhs);
    lv.u[0] = lv.u[1] = lv.d = lv.res = lv.xfer_old = lv.rhs = nullptr;
}

int saena_b200_destroy(saena_b200_ctx *ctx) {
    if (!ctx) return 0;
    cudaSetDevice(ctx->device);
    sb_sync_stream(ctx, ctx->stream);
    sb_sync_stream(ctx, ctx->comm_stream);
    sb_invalidate_graphs(ctx);
    sb_arena_free(ctx);
    sb_f32_free(ctx);
    for (size_t l = 0; l < ctx->levels.size(); ++l) {
        DevLevel &lv = ctx->levels[l];
        sb_free_operator(lv.A); sb_free_operator(lv.P); sb_free_operator(lv.R);
        cudaFree(lv.inv_diag);
        cudaFree(lv.inv_sq_diag);
        free_level_work(lv, l > 0);
    }
    cudaFree(ctx->coarse_A); cudaFree(ctx->coarse_Ainv); cudaFree(ctx->coarse_tmp);
    cudaFree(ctx->ccg_res); cudaFree(ctx->ccg_dir); cudaFree(ctx->ccg_mv);
    cudaFree(ctx->red_partials); cudaFree(ctx->red_counter); cudaFree(ctx->scalars);
    cudaFreeHost(ctx->scalars_host);
    cudaFree(ctx->pcg_r); cudaFree(ctx->pcg_p); cudaFree(ctx->pcg_h); cudaFree(ctx->pcg_u); cudaFree(ctx->pcg_rhs);
    for (int i = 0; i < 4; ++i) cudaFree(ctx->stage[i]);
    cudaFree(ctx->flush_buf);
    cudaFree(ctx->tune_dev);
    cudaFree(ctx->route_t); cudaFree(ctx->route_s);
    sb_block_free(ctx);
    sb_nccl_destroy(ctx);
    cudaEventDestroy(ctx->ev_packed); cudaEventDestroy(ctx->ev_halo);
    cudaEventDestroy(ctx->ev_t0); cudaEventDestroy(ctx->ev_t1);
    cudaStreamDestroy(ctx->stream); cudaStreamDestroy(ctx->comm_stream);
    delete ctx;
    return 0;
}

int saena_b200_upload_operator(saena_b200_ctx *ctx, const saena_b200_operator_desc *desc) {
    if (!ctx || !desc) return 1;
    SB_CUDA(cudaSetDevice(ctx->device));
    return sb_upload_operator(ctx, desc);
}

int saena_b200_upload_band_operator(saena_b200_ctx *ctx, int level, int n, int half_bandwidth, int sliced_only) {
    if (!ctx) return 1;
    SB_CUDA(cudaSetDevice(ctx->device));
    return sb_upload_band_operator(ctx, level, n, half_bandwidth, sliced_only);
}

int saena_b200_upload_level_aux(saena_b200_ctx *ctx, int level, const double *inv_diag, double eig_max,
                                int M_coarse_old, int M_coarse, int n_send, const saena_b200_block *send,
                                int n_recv, const saena_b200_block *recv) {
    if (!ctx) return 1;
    SB_CUDA(cudaSetDevice(ctx->device));
    if (level < 0 || level >= (int)ctx->levels.size() || !ctx->levels[level].A.present)
        SB_FAIL("upload_level_aux: upload A of this level first");
    DevLevel &lv = ctx->levels[level];
    cudaFree(lv.inv_diag);
    lv.inv_diag = nullptr;
    SB_CUDA(cudaMalloc((void **)&lv.inv_diag, sizeof(double) * std::max(lv.M, 1)));
    if (lv.M) SB_CUDA(cudaMemcpy(lv.inv_diag, inv_diag, sizeof(double) * lv.M, cudaMemcpyHostToDevice));
    lv.eig_max = eig_max;
    lv.M_coarse_old = M_coarse_old;
    lv.M_coarse = M_coarse;
    lv.repart.send.assign(send, send + n_send);
    lv.repart.recv.assign(recv, recv + n_recv);
    for (const auto &b : lv.repart.send)
        if (b.peer < 0 || b.peer >= ctx->nranks || b.offset < 0 || b.offset + b.count > M_coarse_old)
            SB_FAIL("upload_level_aux: send block out of range");
    for (const auto &b : lv.repart.recv)
        if (b.peer < 0 || b.peer >= ctx->nranks || b.offset < 0 || b.offset + b.count > M_coarse)
            SB_FAIL("upload_level_aux: recv block out of range");
    lv.aux_set = true;
    ctx->finalized = false;
    return 0;
}

int saena_b200_upload_level_scale(saena_b200_ctx *ctx, int level, const double *inv_sq_diag_orig) {
    if (!ctx) return 1;
    SB_CUDA(cudaSetDevice(ctx->device));
    if (level < 0 || level >= (int)ctx->levels.size() || !ctx->levels[level].A.present)
        SB_FAIL("upload_level_scale: upload A of this level first");
    DevLevel &lv = ctx->levels[level];
    cudaFree(lv.inv_sq_diag);
    lv.inv_sq_diag = nullptr;
    SB_CUDA(cudaMalloc((void **)&lv.inv_sq_diag, sizeof(double) * std::max(lv.M, 1)));
    if (lv.M) SB_CUDA(cudaMemcpy(lv.inv_sq_diag, inv_sq_diag_orig, sizeof(double) * lv.M, cudaMemcpyHostToDevice));
    if (level == 0) ctx->scale = true;
    sb_invalidate_graphs(ctx);
    return 0;
}

}  // extern "C"

// Dense LU with partial pivoting on the host, then the explicit inverse; the device applies
// Ainv with one refinement step against A (vector_ops.cu).  Stands in for SuperLU_DIST's
// factor + pdgssvx solve (saena_object_solve.cpp:117-419, :793-958).  Used by the upload and by
// saena_b200_update_values; the factor's old buffers are released once the new one is computed.
int sb_coarsest_factor(saena_b200_ctx *ctx, int n, int64_t nnz, const int32_t *row, const int32_t *col, const double *val) {
    // coarsest_kernel keeps one n-vector in dynamic shared memory: 4096 doubles = 32 KB, inside the 48 KB default
    if (n < 1 || n > 4096) SB_FAIL("coarsest factor: coarsest level must have 1..4096 rows");
    std::vector<double> A((size_t)n * n, 0.0);
    for (int64_t k = 0; k < nnz; ++k) {
        if (row[k] < 0 || row[k] >= n || col[k] < 0 || col[k] >= n) SB_FAIL("coarsest factor: index out of range");
        A[(size_t)row[k] * n + col[k]] += val[k];
    }
    std::vector<double> LU(A), inv((size_t)n * n, 0.0);
    std::vector<int> piv(n);
    for (int k = 0; k < n; ++k) {
        int p = k;
        double best = fabs(LU[(size_t)k * n + k]);
        for (int i = k + 1; i < n; ++i)
            if (fabs(LU[(size_t)i * n + k]) > best) { best = fabs(LU[(size_t)i * n + k]); p = i; }
        if (best == 0.0) SB_FAIL("coarsest factor: coarsest operator is singular");
        piv[k] = p;
        if (p != k)
            for (int j = 0; j < n; ++j) std::swap(LU[(size_t)k * n + j], LU[(size_t)p * n + j]);
        const double dkk = LU[(size_t)k * n + k];
        for (int i = k + 1; i < n; ++i) {
            const double lik = LU[(size_t)i * n + k] / dkk;
            LU[(size_t)i * n + k] = lik;
            if (lik != 0.0)
                for (int j = k + 1; j < n; ++j) LU[(size_t)i * n + j] -= lik * LU[(size_t)k * n + j];
        }
    }
    std::vector<double> c(n);
    for (int e = 0; e < n; ++e) {  // column e of the inverse
        std::fill(c.begin(), c.end(), 0.0);
        c[e] = 1.0;
        for (int k = 0; k < n; ++k)
            if (piv[k] != k) std::swap(c[k], c[piv[k]]);
        for (int i = 0; i < n; ++i) {
            double s = c[i];
            for (int j = 0; j < i; ++j) s -= LU[(size_t)i * n + j] * c[j];
            c[i] = s;
        }
        for (int i = n - 1; i >= 0; --i) {
            double s = c[i];
            for (int j = i + 1; j < n; ++j) s -= LU[(size_t)i * n + j] * c[j];
            c[i] = s / LU[(size_t)i * n + i];
        }
        for (int i = 0; i < n; ++i) inv[(size_t)i * n + e] = c[i];
    }
    cudaFree(ctx->coarse_A); cudaFree(ctx->coarse_Ainv); cudaFree(ctx->coarse_tmp);
    ctx->coarse_A = ctx->coarse_Ainv = ctx->coarse_tmp = nullptr;
    ctx->coarse_n = 0;
    SB_CUDA(cudaMalloc((void **)&ctx->coarse_A, sizeof(double) * n * n));
    SB_CUDA(cudaMalloc((void **)&ctx->coarse_Ainv, sizeof(double) * n * n));
    SB_CUDA(cudaMalloc((void **)&ctx->coarse_tmp, sizeof(double) * 2 * n));
    SB_CUDA(cudaMemcpy(ctx->coarse_A, A.data(), sizeof(double) * n * n, cudaMemcpyHostToDevice));
    SB_CUDA(cudaMemcpy(ctx->coarse_Ainv, inv.data(), sizeof(double) * n * n, cudaMemcpyHostToDevice));
    ctx->coarse_n = n;
    return 0;
}

extern "C" {

int saena_b200_upload_coarsest(saena_b200_ctx *ctx, int n, int64_t nnz, const int32_t *row, const int32_t *col,
                               const double *val) {
    if (!ctx) return 1;
    SB_CUDA(cudaSetDevice(ctx->device));
    sb_invalidate_graphs(ctx);  // a captured V-cycle's coarsest_kernel node points at the buffers released below
    ctx->finalized = false;
    cudaFree(ctx->coarse_A); cudaFree(ctx->coarse_Ainv); cudaFree(ctx->coarse_tmp);
    ctx->coarse_A = ctx->coarse_Ainv = ctx->coarse_tmp = nullptr;
    ctx->coarse_n = 0;
    if (n == 0) return 0;
    return sb_coarsest_factor(ctx, n, nnz, row, col, val);
}

static int alloc_d(saena_b200_ctx *ctx, double **p, size_t n) {
    *p = nullptr;
    SB_CUDA(cudaMalloc((void **)p, sizeof(double) * std::max<size_t>(n, 1)));
    SB_CUDA(cudaMemset(*p, 0, sizeof(double) * std::max<size_t>(n, 1)));
    return 0;
}

// the two fine-level intermediates of the level route (sb_apply_level_A)
static void route_free(saena_b200_ctx *ctx) {
    cudaFree(ctx->route_t); cudaFree(ctx->route_s);
    ctx->route_t = ctx->route_s = nullptr;
    ctx->route_cap = 0;
}

static int route_alloc(saena_b200_ctx *ctx, int n) {
    if (ctx->route_cap >= n) return 0;
    route_free(ctx);
    SB_TRY(alloc_d(ctx, &ctx->route_t, n));
    SB_TRY(alloc_d(ctx, &ctx->route_s, n));
    ctx->route_cap = n;
    return 0;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// block solve buffers
// ---------------------------------------------------------------------------------------------
static void drop_block_graphs(saena_b200_ctx *ctx) {
    for (size_t i = 0; i < ctx->graphs.size(); ++i)
        if (ctx->graphs[i].k) {
            if (ctx->graphs[i].exec) cudaGraphExecDestroy(ctx->graphs[i].exec);
            ctx->graphs.erase(ctx->graphs.begin() + i);
            --i;
        }
}

void sb_block_free(saena_b200_ctx *ctx) {
    drop_block_graphs(ctx);
    for (DevLevel &lv : ctx->levels) {
        cudaFree(lv.bu[0]); cudaFree(lv.bu[1]); cudaFree(lv.bd); cudaFree(lv.bres); cudaFree(lv.brhs);
        cudaFree(lv.bxfer_old);
        lv.bu[0] = lv.bu[1] = lv.bd = lv.bres = lv.brhs = lv.bxfer_old = nullptr;
        lv.bcur = 0;
    }
    double **vecs[] = {&ctx->blk_r, &ctx->blk_p, &ctx->blk_h, &ctx->blk_u, &ctx->blk_rhs, &ctx->blk_route_t,
                       &ctx->blk_route_s, &ctx->blk_partials, &ctx->blk_scal};
    for (double **v : vecs) { cudaFree(*v); *v = nullptr; }
    cudaFree(ctx->blk_counter); ctx->blk_counter = nullptr;
    cudaFree(ctx->blk_active); ctx->blk_active = nullptr;
    cudaFreeHost(ctx->blk_scal_host); ctx->blk_scal_host = nullptr;
    cudaFreeHost(ctx->blk_active_host); ctx->blk_active_host = nullptr;
    ctx->blk_cap = 0;
    ctx->blk_route_cap = 0;
}

int sb_block_reserve(saena_b200_ctx *ctx, int k) {
    size_t route_rows = 0;   // the largest fine level under a level on the route
    for (size_t l = 1; l < ctx->levels.size(); ++l)
        if (ctx->levels[l].route) route_rows = std::max(route_rows, (size_t)ctx->levels[l - 1].M);
    if (k <= ctx->blk_cap && route_rows * ctx->blk_cap <= ctx->blk_route_cap) return 0;
    const int cap = std::max(k, ctx->blk_cap);
    sb_block_free(ctx);   // also drops every block graph: they point into the buffers being replaced
    const int L = (int)ctx->levels.size();
    bool ok = true;
    auto grab = [&](double **p, size_t n) {
        if (!ok) return;
        ok = cudaMalloc((void **)p, sizeof(double) * std::max<size_t>(n, 1)) == cudaSuccess &&
             cudaMemsetAsync(*p, 0, sizeof(double) * std::max<size_t>(n, 1), ctx->stream) == cudaSuccess;
    };
    for (int l = 0; l < L; ++l) {
        DevLevel &lv = ctx->levels[l];
        const size_t n = (size_t)cap * lv.M;
        grab(&lv.bu[0], n);
        grab(&lv.bu[1], n);
        grab(&lv.bd, n);
        grab(&lv.bres, n);
        if (l > 0) grab(&lv.brhs, n);
        if (l < L - 1 && !lv.repart.identity()) grab(&lv.bxfer_old, (size_t)cap * lv.M_coarse_old);
    }
    const size_t n0 = (size_t)cap * ctx->levels[0].M;
    for (double **v : {&ctx->blk_r, &ctx->blk_p, &ctx->blk_h, &ctx->blk_u, &ctx->blk_rhs}) grab(v, n0);
    if (route_rows) {
        grab(&ctx->blk_route_t, route_rows * cap);
        grab(&ctx->blk_route_s, route_rows * cap);
    }
    grab(&ctx->blk_partials, (size_t)SB_BLOCK_MAX * RED_MAX_BLOCKS);
    grab(&ctx->blk_scal, (size_t)S_COUNT * SB_BLOCK_MAX);
    ok = ok && cudaMalloc((void **)&ctx->blk_counter, sizeof(unsigned int) * SB_BLOCK_MAX) == cudaSuccess &&
         cudaMemsetAsync(ctx->blk_counter, 0, sizeof(unsigned int) * SB_BLOCK_MAX, ctx->stream) == cudaSuccess;
    ok = ok && cudaMalloc((void **)&ctx->blk_active, sizeof(int) * SB_BLOCK_MAX) == cudaSuccess;
    ok = ok && cudaMallocHost((void **)&ctx->blk_scal_host, sizeof(double) * S_COUNT * SB_BLOCK_MAX) == cudaSuccess;
    ok = ok && cudaMallocHost((void **)&ctx->blk_active_host, sizeof(int) * SB_BLOCK_MAX) == cudaSuccess;
    if (!ok) {
        cudaGetLastError();   // an out-of-memory status is not sticky: clear it, the single path is unaffected
        sb_block_free(ctx);
        SB_FAIL("block solve: not enough device memory for the work vectors of " + std::to_string(cap) +
                " right-hand sides");
    }
    ctx->blk_cap = cap;
    ctx->blk_route_cap = route_rows * cap;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// FP32 preconditioner state (saena_b200_set_precond_precision)
// ---------------------------------------------------------------------------------------------
void sb_f32_free(saena_b200_ctx *ctx) {
    for (size_t i = 0; i < ctx->graphs.size(); ++i)
        if (ctx->graphs[i].bits == 32) {
            if (ctx->graphs[i].exec) cudaGraphExecDestroy(ctx->graphs[i].exec);
            ctx->graphs.erase(ctx->graphs.begin() + i);
            --i;
        }
    for (DevLevel &lv : ctx->levels) {
        float **vecs[] = {&lv.u32[0], &lv.u32[1], &lv.d32, &lv.res32, &lv.rhs32, &lv.inv_diag32};
        for (float **v : vecs) { cudaFree(*v); *v = nullptr; }
        for (DevOperator *op : {&lv.A, &lv.P, &lv.R}) {
            float **vals[] = {&op->val32, &op->sell.val32, &op->sellp.val32, &op->sdiag_val32};
            for (float **v : vals) { cudaFree(*v); *v = nullptr; }
        }
    }
    cudaFree(ctx->route32_t); cudaFree(ctx->route32_s);
    ctx->route32_t = ctx->route32_s = nullptr;
}

// nullptr when the hierarchy can run the FP32 preconditioner, else why not: every operator needs an FP32 body
// (spmv_f32.cu) and the V-cycle no FP64-only step
static const char *f32_refusal(const saena_b200_ctx *ctx) {
    if (ctx->nranks != 1 || ctx->detached) return "one rank only";
    if (!ctx->finalized) return "call saena_b200_finalize first";
    if (ctx->scale) return "not on a scaled hierarchy";
    const size_t L = ctx->levels.size();
    for (size_t l = 0; l < L; ++l) {
        const DevLevel &lv = ctx->levels[l];
        if (l + 1 < L && !lv.repart.identity()) return "a level repartitions its coarse vector";
        for (const DevOperator *op : {&lv.A, &lv.P, &lv.R}) {
            if (!op->present) continue;
            if (!op->sends.empty() || !op->recvs.empty() || op->nnz_remote > 0 || op->merged)
                return "an operator has a halo or is in the merged layout";
            if (op->mapping < 0) return "an operator is on streaming row blocks";
        }
    }
    return nullptr;
}

// stored entries of a sliced layout: the last slice offset
static int sliced_entries(saena_b200_ctx *ctx, const SlicedLayout &s, int n_slices, long long *out) {
    SB_CUDA(cudaMemcpy(out, s.ptr + n_slices, sizeof(long long), cudaMemcpyDeviceToHost));
    return 0;
}

static int f32_build(saena_b200_ctx *ctx) {
    bool ok = true;
    auto grab = [&](float **p, size_t n) {
        if (!ok) return;
        ok = cudaMalloc((void **)p, sizeof(float) * std::max<size_t>(n, 1)) == cudaSuccess &&
             cudaMemsetAsync(*p, 0, sizeof(float) * std::max<size_t>(n, 1), ctx->stream) == cudaSuccess;
    };
    // FP32 copy of `n` FP64 values
    auto copy = [&](float **p, const double *src, size_t n) -> int {
        grab(p, n);
        if (ok && n) SB_TRY(sb_convert(ctx, n, src, *p));
        return 0;
    };
    for (DevLevel &lv : ctx->levels) {
        // every work vector sized from the level's rows, as its FP64 twin
        for (float **v : {&lv.u32[0], &lv.u32[1], &lv.d32, &lv.res32, &lv.rhs32}) grab(v, lv.M);
        SB_TRY(copy(&lv.inv_diag32, lv.inv_diag, lv.M));
        for (DevOperator *op : {&lv.A, &lv.P, &lv.R}) {
            if (!op->present || !ok) continue;
            long long n = 0;
            if (op->mapping == SB_MAPPING_SELL) {
                SB_TRY(sliced_entries(ctx, op->sell, (op->M + 31) / 32, &n));
                SB_TRY(copy(&op->sell.val32, op->sell.val, n));
            } else if (op->mapping == SB_MAPPING_SELLP) {
                SB_TRY(sliced_entries(ctx, op->sellp, (op->M + 255) / 256 * 8, &n));
                SB_TRY(copy(&op->sellp.val32, op->sellp.val, n));
            } else if (op->mapping == SB_MAPPING_SYMDIAG) {
                SB_TRY(copy(&op->sdiag_val32, op->sdiag_val, (size_t)op->sdiag.nd * op->M));
            } else {
                SB_TRY(copy(&op->val32, op->val, op->nnz_local));
            }
        }
    }
    if (ctx->route_cap > 0) {
        grab(&ctx->route32_t, ctx->route_cap);
        grab(&ctx->route32_s, ctx->route_cap);
    }
    if (!ok) {
        cudaGetLastError();   // an out-of-memory status is not sticky
        SB_FAIL("set_precond_precision: not enough device memory for the FP32 copies");
    }
    return sb_sync_stream(ctx, ctx->stream);
}

int sb_f32_sync(saena_b200_ctx *ctx) {
    if (ctx->precond_bits != 32 || !ctx->f32_stale) return 0;
    sb_f32_free(ctx);   // the copies of layouts no longer in use, and every captured FP32 V-cycle
    const char *why = f32_refusal(ctx);
    const int rc = why ? 1 : f32_build(ctx);
    if (rc) {
        sb_f32_free(ctx);
        ctx->precond_bits = 64;
        if (why) SB_FAIL(std::string("precision 32: ") + why + "; the preconditioner stays FP64");
        return rc;
    }
    ctx->f32_stale = false;
    return 0;
}

extern "C" {

int saena_b200_set_precond_precision(saena_b200_ctx *ctx, int bits) {
    if (!ctx) return 1;
    SB_CUDA(cudaSetDevice(ctx->device));
    if (bits != 32 && bits != 64) SB_FAIL("set_precond_precision: bits must be 32 or 64");
    if (bits == 64) {
        sb_f32_free(ctx);
        ctx->precond_bits = 64;
        return 0;
    }
    if (ctx->precond_bits != 32) {
        ctx->precond_bits = 32;
        ctx->f32_stale = true;
    }
    return sb_f32_sync(ctx);
}

int saena_b200_get_precond_precision(const saena_b200_ctx *ctx) { return ctx ? ctx->precond_bits : 0; }

int saena_b200_finalize(saena_b200_ctx *ctx) {
    if (!ctx) return 1;
    SB_CUDA(cudaSetDevice(ctx->device));
    const int L = (int)ctx->levels.size();
    if (L == 0) SB_FAIL("finalize: no level uploaded");
    sb_invalidate_graphs(ctx);
    // the operators may have been replaced: every level starts on its stored A (the route is chosen again by
    // saena_b200_autotune_mapping or saena_b200_set_level_route)
    for (DevLevel &lv : ctx->levels) {
        lv.route = false;
        lv.route_ms[0] = lv.route_ms[1] = 0.f;
    }
    route_free(ctx);
    sb_block_free(ctx);
    sb_f32_free(ctx);
    ctx->precond_bits = 64;
    SB_TRY(sb_arena_build(ctx));  // ghost buffers of every operator, one allocation (p2p_halo.cu)
    for (int l = 0; l < L; ++l) {
        DevLevel &lv = ctx->levels[l];
        if (!lv.A.present) SB_FAIL("finalize: a level has no A");
        if (!lv.aux_set) SB_FAIL("finalize: upload_level_aux missing for a level");
        if (l < L - 1) {
            if (!lv.P.present || !lv.R.present) SB_FAIL("finalize: P/R missing on a non-coarsest level");
            DevLevel &cl = ctx->levels[l + 1];
            if (lv.P.M != lv.M || lv.R.n_local_cols != lv.M) SB_FAIL("finalize: P rows / R columns != A rows");
            if (lv.R.M != lv.M_coarse_old || lv.P.n_local_cols != lv.M_coarse_old)
                SB_FAIL("finalize: R rows / P columns != M_coarse_old");
            if (cl.M != lv.M_coarse) SB_FAIL("finalize: coarse A rows != M_coarse");
            if (lv.repart.identity() && lv.M_coarse_old != lv.M_coarse)
                SB_FAIL("finalize: partitions differ but no repartition plan was given");
        }
        free_level_work(lv, l > 0);
        SB_TRY(alloc_d(ctx, &lv.u[0], lv.M));
        SB_TRY(alloc_d(ctx, &lv.u[1], lv.M));
        SB_TRY(alloc_d(ctx, &lv.d, lv.M));
        SB_TRY(alloc_d(ctx, &lv.res, lv.M));
        if (l > 0) SB_TRY(alloc_d(ctx, &lv.rhs, lv.M));
        if (l < L - 1 && !lv.repart.identity()) SB_TRY(alloc_d(ctx, &lv.xfer_old, lv.M_coarse_old));
        lv.cur = 0;
        SB_TRY(sb_prepare_operator(ctx, lv.A));
        SB_TRY(sb_prepare_operator(ctx, lv.P));
        SB_TRY(sb_prepare_operator(ctx, lv.R));
    }
    if (ctx->coarse_n != 0 && ctx->levels[L - 1].M > 0 && ctx->coarse_n != ctx->levels[L - 1].M)
        SB_FAIL("finalize: the coarsest factor's size differs from the coarsest level's rows");
    // (no factor at all is accepted: a lone operator uploaded for matvec only; any V-cycle then fails loudly)
    const int n0 = ctx->levels[0].M;
    cudaFree(ctx->pcg_r); cudaFree(ctx->pcg_p); cudaFree(ctx->pcg_h); cudaFree(ctx->pcg_u); cudaFree(ctx->pcg_rhs);
    SB_TRY(alloc_d(ctx, &ctx->pcg_r, n0));
    SB_TRY(alloc_d(ctx, &ctx->pcg_p, n0));
    SB_TRY(alloc_d(ctx, &ctx->pcg_h, n0));
    SB_TRY(alloc_d(ctx, &ctx->pcg_u, n0));
    SB_TRY(alloc_d(ctx, &ctx->pcg_rhs, n0));
    ctx->pcg_cap = n0;
    ctx->finalized = true;
    return 0;
}

}  // extern "C"

// cudaStreamSynchronize with a watchdog: the host polls the stream and gives up after sync_timeout_s -- a peer process
// that died inside a collective, or any other stall the device-side deadlines do not cover, becomes an error status
// instead of a process that never returns (the reference: print + MPI_Abort, src/saena_object_solve.cpp:1012-1013).
int sb_sync_stream(saena_b200_ctx *ctx, cudaStream_t s) {
    if (ctx->nranks == 1 || ctx->sync_timeout_s <= 0.0) {
        SB_CUDA(cudaStreamSynchronize(s));
        return 0;
    }
    struct timespec t0;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    for (unsigned int n = 0;; ++n) {
        const cudaError_t q = cudaStreamQuery(s);
        if (q == cudaSuccess) return 0;
        if (q != cudaErrorNotReady) {
            ctx->error = std::string("cudaStreamQuery: ") + cudaGetErrorString(q);
            return 1;
        }
        if ((n & 1023u) == 1023u) {
            struct timespec t1;
            clock_gettime(CLOCK_MONOTONIC, &t1);
            const double el = (double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec);
            if (el > ctx->sync_timeout_s) {
                ctx->faulted = true;
                ctx->error = "rank " + std::to_string(ctx->rank) + ": the device did not finish within " +
                             std::to_string((int)ctx->sync_timeout_s) +
                             " s (a peer that left a collective? SAENA_B200_SYNC_TIMEOUT_S); the context is unusable";
                return 1;
            }
        }
    }
}

// The fault words arrive with every sb_read_scalars; entry points that do not read scalars fetch them here.
int sb_check_fault(saena_b200_ctx *ctx) {
    if (ctx->nranks == 1) return 0;
    const unsigned long long *f = (const unsigned long long *)(ctx->scalars_host + S_COUNT);
    if (!ctx->faulted && f[0] == 0ull) {
        SB_CUDA(cudaMemcpyAsync(ctx->scalars_host + S_COUNT, ctx->scalars + S_COUNT, sizeof(double) * S_FAULT_WORDS,
                                cudaMemcpyDeviceToHost, ctx->stream));
        SB_TRY(sb_sync_stream(ctx, ctx->stream));
    }
    if (f[0] != 0ull) {
        const int what = (int)(f[0] & 0xffull), op_id = (int)((f[0] >> 8) & 0xffffffull), slot = (int)(f[0] >> 32);
        ctx->faulted = true;
        ctx->error = "rank " + std::to_string(ctx->rank) + ": halo exchange timed out after " +
                     std::to_string(ctx->halo_timeout_ns / 1000000ull) + " ms on level " + std::to_string(op_id / 3) +
                     " operator " + "APR"[op_id % 3] + ": waited for the '" +
                     (what == 1 ? "consumed" : "arrived") + "' counter of neighbour slot " + std::to_string(slot) +
                     " to reach " + std::to_string(f[1]) + ", saw " + std::to_string(f[2]) +
                     " (SAENA_B200_HALO_TIMEOUT_MS; results of this call are invalid)";
        return 1;
    }
    if (ctx->faulted) {
        if (ctx->error.empty()) ctx->error = "an earlier call of this context timed out (saena_b200_clear_fault)";
        return 1;
    }
    return 0;
}

static __global__ void fault_flag_kernel(const unsigned long long *fault, double *out) { *out = fault[0] != 0ull ? 1.0 : 0.0; }

int sb_agree_fault(saena_b200_ctx *ctx) {
    if (ctx->nranks == 1 || ctx->detached) return 0;
    fault_flag_kernel<<<1, 1, 0, ctx->stream>>>(ctx->fault_dev, ctx->scalars + S_AGREE);
    SB_CUDA(cudaGetLastError());
    SB_TRY(sb_allreduce_sum(ctx, ctx->scalars + S_AGREE, 1, ctx->stream));
    SB_TRY(sb_read_scalars(ctx));
    SB_TRY(sb_check_fault(ctx));
    if (ctx->scalars_host[S_AGREE] > 0.0) {
        ctx->faulted = true;
        ctx->error = "rank " + std::to_string(ctx->rank) + ": the halo exchange of " +
                     std::to_string((int)ctx->scalars_host[S_AGREE]) +
                     " peer rank(s) timed out during this call (results are invalid on every rank)";
        return 1;
    }
    return 0;
}

extern "C" {

// After a timed-out exchange every rank's counters are out of step: the peer-memory transport stays off until the
// next saena_b200_p2p_import.  Clears the fault so that the context can go on over NCCL (collective by contract: all
// ranks call it, then saena_b200_p2p_enable(ctx, 0)).
int saena_b200_clear_fault(saena_b200_ctx *ctx) {
    if (!ctx) return 1;
    SB_CUDA(cudaSetDevice(ctx->device));
    SB_TRY(sb_sync_stream(ctx, ctx->stream));
    SB_TRY(sb_sync_stream(ctx, ctx->comm_stream));
    SB_CUDA(cudaMemset(ctx->fault_dev, 0, sizeof(unsigned long long) * S_FAULT_WORDS));
    memset(ctx->scalars_host + S_COUNT, 0, sizeof(double) * S_FAULT_WORDS);
    ctx->faulted = false;
    ctx->error.clear();
    sb_invalidate_graphs(ctx);
    return 0;
}

// halo_timeout_ms: deadline of every device-side wait of the exchange; sync_timeout_s: watchdog of the blocking host
// waits (<= 0: none).  Negative halo_timeout_ms leaves that value as it is.
int saena_b200_set_timeouts(saena_b200_ctx *ctx, double halo_timeout_ms, double sync_timeout_s) {
    if (!ctx) return 1;
    if (halo_timeout_ms >= 0.0) ctx->halo_timeout_ns = (unsigned long long)(halo_timeout_ms * 1e6);
    ctx->sync_timeout_s = sync_timeout_s;
    sb_invalidate_graphs(ctx);   // captured kernel nodes carry the old deadline in their arguments
    return 0;
}

int saena_b200_fault_status(saena_b200_ctx *ctx) {
    if (!ctx) return 1;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return 1;
    return sb_check_fault(ctx);
}

#define SB_ENTER()                                                        \
    if (!ctx) return 1;                                                   \
    SB_CUDA(cudaSetDevice(ctx->device));                                  \
    if (!ctx->finalized) SB_FAIL("call saena_b200_finalize first");       \
    if (ctx->faulted) return sb_check_fault(ctx)

static int stage_buf(saena_b200_ctx *ctx, int i, size_t n) {
    if (ctx->stage_cap[i] < n) {
        cudaFree(ctx->stage[i]);
        ctx->stage[i] = nullptr;
        ctx->stage_cap[i] = 0;
        SB_CUDA(cudaMalloc((void **)&ctx->stage[i], sizeof(double) * std::max<size_t>(n, 1)));
        ctx->stage_cap[i] = n;
    }
    return 0;
}
extern "C++" {   // templates, inside the extern "C" block of the entry points
template <typename T>
static int h2d(saena_b200_ctx *ctx, T *dst, const T *src, size_t n) {
    if (n) SB_CUDA(cudaMemcpyAsync(dst, src, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    return 0;
}
template <typename T>
static int d2h(saena_b200_ctx *ctx, T *dst, const T *src, size_t n) {
    if (n) SB_CUDA(cudaMemcpyAsync(dst, src, n * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
    SB_TRY(sb_sync_stream(ctx, ctx->stream));
    return sb_check_fault(ctx);   // every host-buffer entry point ends here: a timed-out exchange is an error status
}

static DevOperator *get_op(saena_b200_ctx *ctx, int level, int kind) {
    if (level < 0 || level >= (int)ctx->levels.size()) return nullptr;
    DevOperator *op = &ctx->levels[level].op(kind);
    return op->present ? op : nullptr;
}

// what the solve applies for (level, kind): A through sb_apply_level_A (the route on a route level)
template <typename V>
static int apply_kind(saena_b200_ctx *ctx, int level, int kind, const V *x, int epi, const EpiArgsT<V> &e) {
    if (kind == SAENA_B200_KIND_A) return sb_apply_level_A(ctx, level, x, epi, e);
    return sb_apply(ctx, *get_op(ctx, level, kind), x, epi, e);
}
}  // extern "C++"

// ---------------------------------------------------------------------------------------------
// Krylov drivers (device-resident vectors; one host read of <r,r> per iteration for the stop test)
// ---------------------------------------------------------------------------------------------
static void push_hist(double v, double *hist, int cap, int &n) {
    if (hist && n < cap) hist[n] = sqrt(v);
    ++n;
}

// rho = M^-1 r from a zero iterate into level 0's u[cur].  Precision 32: r rounded into level 0's FP32 rhs, the FP32
// V-cycle, its iterate widened into u[0] (cur = 0); the Krylov loop around it stays FP64.
static int precondition(saena_b200_ctx *ctx, int smoother, int pre, int post, const double *r) {
    if (ctx->precond_bits != 32) return sb_vcycle_from_zero(ctx, smoother, pre, post, r);
    SB_TRY(sb_f32_sync(ctx));
    DevLevel &l0 = ctx->levels[0];
    SB_TRY(sb_convert(ctx, l0.M, r, l0.rhs32));
    SB_TRY(sb_vcycle_from_zero(ctx, smoother, pre, post, (const float *)l0.rhs32));
    SB_TRY(sb_convert(ctx, l0.M, l0.u32[l0.cur], l0.u[0]));
    l0.cur = 0;
    return 0;
}

static int pcg_device(saena_b200_ctx *ctx, const double *rhs, double *u, int max_iter, double tol, int smoother,
                      int pre, int post, int *iters, double *hist, int hist_cap, int *hist_len) {
    DevLevel &l0 = ctx->levels[0];
    const int n = l0.M;
    const int max_level = (int)ctx->levels.size() - 1;
    double *r = ctx->pcg_r, *p = ctx->pcg_p, *h = ctx->pcg_h;
    int nh = 0;
    // u = 0 (:2482); r = A u - rhs = -rhs (:2496); init_dot = <r,r> (:2501)
    SB_TRY(sb_fill_zero(ctx, u, n));
    SB_TRY(sb_negate_copy(ctx, n, rhs, r));
    SB_TRY(sb_dot(ctx, r, r, n, S_RR));
    SB_TRY(sb_read_scalars(ctx));
    const double init_dot = ctx->scalars_host[S_RR];
    double current_dot = init_dot;
    push_hist(init_dot, hist, hist_cap, nh);
    int i = 0;
    if (max_level == 0) {
        // :2507-2521 direct solver only: u = A^-1 rhs
        l0.cur = 0;
        SB_TRY(sb_vcycle(ctx, 0, smoother, pre, post, rhs, true));
        if (n) SB_CUDA(cudaMemcpyAsync(u, l0.u[l0.cur], sizeof(double) * n, cudaMemcpyDeviceToDevice, ctx->stream));
        EpiArgs e{};
        e.rhs = rhs;
        e.out = r;
        SB_TRY(sb_apply(ctx, l0.A, u, EPI_RESIDUAL, e));
        SB_TRY(sb_dot(ctx, r, r, n, S_RR));
        SB_TRY(sb_read_scalars(ctx));
        push_hist(ctx->scalars_host[S_RR], hist, hist_cap, nh);
        if (ctx->scale) SB_TRY(sb_scale_vector(ctx, n, u, l0.inv_sq_diag));  // :2517-2519
        *iters = 1;
        *hist_len = nh;
        return 0;
    }
    // rho = 0; vcycle(rho, r) (:2535-2537); rho lives in level 0's iterate buffers
    SB_TRY(precondition(ctx, smoother, pre, post, r));
    // p = rho (:2554)
    if (n) SB_CUDA(cudaMemcpyAsync(p, l0.u[l0.cur], sizeof(double) * n, cudaMemcpyDeviceToDevice, ctx->stream));
    const double THRSHLD = init_dot * tol * tol;  // :2558
    SB_TRY(sb_dot(ctx, r, l0.u[l0.cur], n, S_RHO_RES));  // first <r,rho> (:2580)
    for (i = 0; i < max_iter; i++) {
        SbRange it_range(ctx, "pcg iteration");
        EpiArgs e{};
        e.out = h;
        { SbRange rg(ctx, "L0matvec"); SB_TRY(sb_apply(ctx, l0.A, p, EPI_PLAIN, e)); }  // h = A p (:2571)
        { SbRange rg(ctx, "dots"); SB_TRY(sb_dot(ctx, p, h, n, S_PDOTH)); }             // :2581
        SB_TRY(sb_pcg_update(ctx, n, u, r, p, h));     // :2588-2603
        SB_TRY(sb_read_scalars(ctx));
        current_dot = ctx->scalars_host[S_RR];
        push_hist(current_dot, hist, hist_cap, nh);
        if (!(current_dot >= THRSHLD)) break;          // :2620 (NaN also stops)
        { SbRange rg(ctx, "vcycle_pCG"); SB_TRY(precondition(ctx, smoother, pre, post, r)); }  // :2640-2641
        SB_TRY(sb_dot(ctx, r, l0.u[l0.cur], n, S_BETA_NUM));      // :2655
        SB_TRY(sb_pcg_p_update(ctx, n, p, l0.u[l0.cur]));          // :2662-2667
    }
    if (i == max_iter) i--;  // :2673-2674
    if (ctx->scale) SB_TRY(sb_scale_vector(ctx, n, u, l0.inv_sq_diag));  // :2709-2711
    *iters = i + 1;          // :2678-2682
    *hist_len = nh;
    (void)current_dot;
    return 0;
}

int saena_b200_solve_pcg_dev(saena_b200_ctx *ctx, const double *rhs_dev, double *u_dev, int max_iter, double tol,
                             int smoother, int pre, int post, int *iters, double *hist, int hist_cap,
                             int *hist_len) {
    SB_ENTER();
    SB_TRY(pcg_device(ctx, rhs_dev, u_dev, max_iter, tol, smoother, pre, post, iters, hist, hist_cap, hist_len));
    SB_TRY(sb_sync_stream(ctx, ctx->stream));
    return sb_agree_fault(ctx);
}

int saena_b200_solve_pcg(saena_b200_ctx *ctx, const double *rhs, double *u, int max_iter, double tol, int smoother,
                         int pre, int post, int *iters, double *hist, int hist_cap, int *hist_len) {
    SB_ENTER();
    const int n = ctx->levels[0].M;
    SB_TRY(h2d(ctx, ctx->pcg_rhs, rhs, n));
    SB_TRY(pcg_device(ctx, ctx->pcg_rhs, ctx->pcg_u, max_iter, tol, smoother, pre, post, iters, hist, hist_cap,
                      hist_len));
    SB_TRY(sb_agree_fault(ctx));
    SB_TRY(d2h(ctx, u, ctx->pcg_u, n));
    return 0;
}

int saena_b200_solve_vcycle(saena_b200_ctx *ctx, const double *rhs, double *u, int max_iter, double tol,
                            int smoother, int pre, int post, int *iters, double *hist, int hist_cap,
                            int *hist_len) {
    SB_ENTER();
    DevLevel &l0 = ctx->levels[0];
    const int n = l0.M;
    double *r = ctx->pcg_r;
    int nh = 0;
    SB_TRY(h2d(ctx, ctx->pcg_rhs, rhs, n));
    const double *b = ctx->pcg_rhs;
    l0.cur = 0;
    SB_TRY(sb_fill_zero(ctx, l0.u[0], n));
    SB_TRY(sb_negate_copy(ctx, n, b, r));
    SB_TRY(sb_dot(ctx, r, r, n, S_RR));
    SB_TRY(sb_read_scalars(ctx));
    const double init_dot = ctx->scalars_host[S_RR];
    push_hist(init_dot, hist, hist_cap, nh);
    const double THRSHLD = init_dot * tol * tol;
    int i = 0;
    for (; i < max_iter; ++i) {
        SB_TRY(sb_vcycle(ctx, 0, smoother, pre, post, b, i == 0));  // u carries over between cycles
        EpiArgs e{};
        e.rhs = b;
        e.out = r;
        SB_TRY(sb_apply(ctx, l0.A, l0.u[l0.cur], EPI_RESIDUAL, e));
        SB_TRY(sb_dot(ctx, r, r, n, S_RR));
        SB_TRY(sb_read_scalars(ctx));
        push_hist(ctx->scalars_host[S_RR], hist, hist_cap, nh);
        if (!(ctx->scalars_host[S_RR] >= THRSHLD)) break;
    }
    if (i == max_iter) --i;
    if (ctx->scale) SB_TRY(sb_scale_vector(ctx, n, l0.u[l0.cur], l0.inv_sq_diag));  // :2000-2002
    *iters = i + 1;
    *hist_len = nh;
    SB_TRY(sb_agree_fault(ctx));
    SB_TRY(d2h(ctx, u, l0.u[l0.cur], n));
    return 0;
}

// saena_object::solve_smoother (src/saena_object_solve.cpp:2017-2117; reached from saena::amg::solve_smoother,
// src/saena.cpp:751-758): the smoother alone as a stationary iteration -- `pre` sweeps (:2074), residual and <r,r>
// (:2075-2076), the solvers' stop rule (:2080) -- on level 0.  Every sweep is the fused one-pass kernel of the V-cycle.
int saena_b200_solve_smoother(saena_b200_ctx *ctx, const double *rhs, double *u, int max_iter, double tol,
                              int smoother, int pre, int post, int *iters, double *hist, int hist_cap,
                              int *hist_len) {
    SB_ENTER();
    (void)post;
    DevLevel &l0 = ctx->levels[0];
    const int n = l0.M;
    double *r = ctx->pcg_r;
    int nh = 0;
    SB_TRY(h2d(ctx, ctx->pcg_rhs, rhs, n));
    const double *b = ctx->pcg_rhs;
    l0.cur = 0;
    SB_TRY(sb_fill_zero(ctx, l0.u[0], n));      // :2051
    SB_TRY(sb_negate_copy(ctx, n, b, r));       // :2061 with u = 0
    SB_TRY(sb_dot(ctx, r, r, n, S_RR));
    SB_TRY(sb_read_scalars(ctx));
    const double init_dot = ctx->scalars_host[S_RR];
    push_hist(init_dot, hist, hist_cap, nh);
    const double THRSHLD = init_dot * tol * tol;  // :2069
    int i = 0;
    for (; i < max_iter; ++i) {
        SB_TRY(sb_smooth(ctx, 0, smoother, pre, b, i == 0));  // the first sweep starts from the zero iterate
        EpiArgs e{};
        e.rhs = b;
        e.out = r;
        SB_TRY(sb_apply(ctx, l0.A, l0.u[l0.cur], EPI_RESIDUAL, e));
        SB_TRY(sb_dot(ctx, r, r, n, S_RR));
        SB_TRY(sb_read_scalars(ctx));
        push_hist(ctx->scalars_host[S_RR], hist, hist_cap, nh);
        if (!(ctx->scalars_host[S_RR] >= THRSHLD)) break;     // :2080
    }
    if (i == max_iter) --i;                                   // :2086-2087
    if (ctx->scale) SB_TRY(sb_scale_vector(ctx, n, l0.u[l0.cur], l0.inv_sq_diag));  // :2100-2102
    *iters = i + 1;
    *hist_len = nh;
    SB_TRY(sb_agree_fault(ctx));
    SB_TRY(d2h(ctx, u, l0.u[l0.cur], n));
    return 0;
}

// Unpreconditioned CG (saena_object_solve.cpp:2119-2386, sign convention r = A u - rhs,
// u -= alpha p).  The reference's pointer aliasing bug at :2311 is not replicated (SURVEY P3).
int saena_b200_solve_cg(saena_b200_ctx *ctx, const double *rhs, double *u, int max_iter, double tol, int *iters,
                        double *hist, int hist_cap, int *hist_len) {
    SB_ENTER();
    DevLevel &l0 = ctx->levels[0];
    const int n = l0.M;
    double *r = ctx->pcg_r, *p = ctx->pcg_p, *h = ctx->pcg_h, *x = ctx->pcg_u;
    int nh = 0;
    SB_TRY(h2d(ctx, ctx->pcg_rhs, rhs, n));
    SB_TRY(sb_fill_zero(ctx, x, n));
    SB_TRY(sb_negate_copy(ctx, n, ctx->pcg_rhs, r));
    SB_TRY(sb_dot(ctx, r, r, n, S_RHO_RES));  // <r,r> plays rho_res
    SB_TRY(sb_read_scalars(ctx));
    const double init_dot = ctx->scalars_host[S_RHO_RES];
    push_hist(init_dot, hist, hist_cap, nh);
    if (n) SB_CUDA(cudaMemcpyAsync(p, r, sizeof(double) * n, cudaMemcpyDeviceToDevice, ctx->stream));
    const double THRSHLD = init_dot * tol * tol;
    int i = 0;
    for (; i < max_iter; ++i) {
        EpiArgs e{};
        e.out = h;
        SB_TRY(sb_apply(ctx, l0.A, p, EPI_PLAIN, e));
        SB_TRY(sb_dot(ctx, p, h, n, S_PDOTH));
        SB_TRY(sb_pcg_update(ctx, n, x, r, p, h));  // alpha = <r,r>/<p,Ap>; writes S_RR
        SB_TRY(sb_read_scalars(ctx));
        push_hist(ctx->scalars_host[S_RR], hist, hist_cap, nh);
        if (!(ctx->scalars_host[S_RR] >= THRSHLD)) break;
        SB_TRY(sb_cg_p_update(ctx, n, p, r, S_RR, S_RHO_RES));  // beta = <r,r>_new / <r,r>_old
        SB_CUDA(cudaMemcpyAsync(ctx->scalars + S_RHO_RES, ctx->scalars + S_RR, sizeof(double),
                                cudaMemcpyDeviceToDevice, ctx->stream));
    }
    if (i == max_iter) --i;
    *iters = i + 1;
    *hist_len = nh;
    SB_TRY(sb_agree_fault(ctx));
    SB_TRY(d2h(ctx, u, x, n));
    return 0;
}

// ---------------------------------------------------------------------------------------------
// per-operator hooks
// ---------------------------------------------------------------------------------------------
int saena_b200_matvec(saena_b200_ctx *ctx, int level, int kind, const double *v, double *w) {
    SB_ENTER();
    DevOperator *op = get_op(ctx, level, kind);
    if (!op) SB_FAIL("matvec: no such operator");
    SB_TRY(stage_buf(ctx, 0, op->n_local_cols));
    SB_TRY(stage_buf(ctx, 1, op->M));
    SB_TRY(h2d(ctx, ctx->stage[0], v, op->n_local_cols));
    EpiArgs e{};
    e.out = ctx->stage[1];
    SB_TRY(apply_kind(ctx, level, kind, ctx->stage[0], EPI_PLAIN, e));
    SB_TRY(d2h(ctx, w, ctx->stage[1], op->M));
    return 0;
}

int saena_b200_residual(saena_b200_ctx *ctx, int level, const double *u, const double *rhs, double *res) {
    SB_ENTER();
    DevOperator *op = get_op(ctx, level, SAENA_B200_KIND_A);
    if (!op) SB_FAIL("residual: no such level");
    for (int i = 0; i < 3; ++i) SB_TRY(stage_buf(ctx, i, op->M));
    SB_TRY(h2d(ctx, ctx->stage[0], u, op->M));
    SB_TRY(h2d(ctx, ctx->stage[1], rhs, op->M));
    EpiArgs e{};
    e.rhs = ctx->stage[1];
    e.out = ctx->stage[2];
    SB_TRY(sb_apply_level_A(ctx, level, ctx->stage[0], EPI_RESIDUAL, e));
    SB_TRY(d2h(ctx, res, ctx->stage[2], op->M));
    return 0;
}

int saena_b200_smooth(saena_b200_ctx *ctx, int level, int smoother, int iters, double *u, const double *rhs) {
    SB_ENTER();
    if (level < 0 || level >= (int)ctx->levels.size()) SB_FAIL("smooth: no such level");
    DevLevel &lv = ctx->levels[level];
    SB_TRY(stage_buf(ctx, 1, lv.M));
    lv.cur = 0;
    SB_TRY(h2d(ctx, lv.u[0], u, lv.M));
    SB_TRY(h2d(ctx, ctx->stage[1], rhs, lv.M));
    SB_TRY(sb_smooth(ctx, level, smoother, iters, ctx->stage[1], false));
    SB_TRY(d2h(ctx, u, lv.u[lv.cur], lv.M));
    return 0;
}

int saena_b200_vcycle(saena_b200_ctx *ctx, int level, int smoother, int pre, int post, double *u,
                      const double *rhs) {
    SB_ENTER();
    if (level < 0 || level >= (int)ctx->levels.size()) SB_FAIL("vcycle: no such level");
    DevLevel &lv = ctx->levels[level];
    SB_TRY(stage_buf(ctx, 1, lv.M));
    lv.cur = 0;
    SB_TRY(h2d(ctx, lv.u[0], u, lv.M));
    SB_TRY(h2d(ctx, ctx->stage[1], rhs, lv.M));
    SB_TRY(sb_vcycle(ctx, level, smoother, pre, post, ctx->stage[1], false));
    SB_TRY(d2h(ctx, u, lv.u[lv.cur], lv.M));
    return 0;
}

int saena_b200_coarsest_solve(saena_b200_ctx *ctx, const double *rhs, double *u) {
    SB_ENTER();
    const int n = ctx->coarse_n;
    SB_TRY(stage_buf(ctx, 0, n));
    SB_TRY(stage_buf(ctx, 1, n));
    SB_TRY(h2d(ctx, ctx->stage[0], rhs, n));
    SB_TRY(sb_coarsest_apply(ctx, ctx->stage[0], ctx->stage[1]));
    SB_TRY(d2h(ctx, u, ctx->stage[1], n));
    return 0;
}

int saena_b200_dot(saena_b200_ctx *ctx, const double *a, const double *b, int n, double *out) {
    SB_ENTER();
    SB_TRY(stage_buf(ctx, 0, n));
    SB_TRY(stage_buf(ctx, 1, n));
    SB_TRY(h2d(ctx, ctx->stage[0], a, n));
    SB_TRY(h2d(ctx, ctx->stage[1], b, n));
    SB_TRY(sb_dot(ctx, ctx->stage[0], ctx->stage[1], n, S_TMP));
    SB_TRY(sb_read_scalars(ctx));
    *out = ctx->scalars_host[S_TMP];
    return sb_check_fault(ctx);
}

// ---------------------------------------------------------------------------------------------
// FP32 hooks: the per-operator hooks above on the FP32 copies and vectors (precision 32 only); staged through the
// same buffers, which hold n floats where they hold n doubles
// ---------------------------------------------------------------------------------------------
#define SB_ENTER_F32(name)                                                                       \
    SB_ENTER();                                                                                  \
    if (ctx->precond_bits != 32) SB_FAIL(name ": call saena_b200_set_precond_precision(ctx, 32) first"); \
    SB_TRY(sb_f32_sync(ctx))

static float *stage32(saena_b200_ctx *ctx, int i) { return (float *)ctx->stage[i]; }

int saena_b200_matvec_f32(saena_b200_ctx *ctx, int level, int kind, const float *v, float *w) {
    SB_ENTER_F32("matvec_f32");
    DevOperator *op = get_op(ctx, level, kind);
    if (!op) SB_FAIL("matvec_f32: no such operator");
    SB_TRY(stage_buf(ctx, 0, op->n_local_cols));
    SB_TRY(stage_buf(ctx, 1, op->M));
    SB_TRY(h2d(ctx, stage32(ctx, 0), v, op->n_local_cols));
    EpiArgs32 e{};
    e.out = stage32(ctx, 1);
    SB_TRY(apply_kind(ctx, level, kind, (const float *)stage32(ctx, 0), EPI_PLAIN, e));
    return d2h(ctx, w, stage32(ctx, 1), op->M);
}

int saena_b200_residual_f32(saena_b200_ctx *ctx, int level, const float *u, const float *rhs, float *res) {
    SB_ENTER_F32("residual_f32");
    DevOperator *op = get_op(ctx, level, SAENA_B200_KIND_A);
    if (!op) SB_FAIL("residual_f32: no such level");
    for (int i = 0; i < 3; ++i) SB_TRY(stage_buf(ctx, i, op->M));
    SB_TRY(h2d(ctx, stage32(ctx, 0), u, op->M));
    SB_TRY(h2d(ctx, stage32(ctx, 1), rhs, op->M));
    EpiArgs32 e{};
    e.rhs = stage32(ctx, 1);
    e.out = stage32(ctx, 2);
    SB_TRY(sb_apply_level_A(ctx, level, (const float *)stage32(ctx, 0), EPI_RESIDUAL, e));
    return d2h(ctx, res, stage32(ctx, 2), op->M);
}

int saena_b200_smooth_f32(saena_b200_ctx *ctx, int level, int smoother, int iters, float *u, const float *rhs) {
    SB_ENTER_F32("smooth_f32");
    if (level < 0 || level >= (int)ctx->levels.size()) SB_FAIL("smooth_f32: no such level");
    DevLevel &lv = ctx->levels[level];
    SB_TRY(stage_buf(ctx, 1, lv.M));
    lv.cur = 0;
    SB_TRY(h2d(ctx, lv.u32[0], u, lv.M));
    SB_TRY(h2d(ctx, stage32(ctx, 1), rhs, lv.M));
    SB_TRY(sb_smooth(ctx, level, smoother, iters, (const float *)stage32(ctx, 1), false));
    return d2h(ctx, u, lv.u32[lv.cur], lv.M);
}

int saena_b200_vcycle_f32(saena_b200_ctx *ctx, int level, int smoother, int pre, int post, float *u, const float *rhs) {
    SB_ENTER_F32("vcycle_f32");
    if (level < 0 || level >= (int)ctx->levels.size()) SB_FAIL("vcycle_f32: no such level");
    DevLevel &lv = ctx->levels[level];
    SB_TRY(stage_buf(ctx, 1, lv.M));
    lv.cur = 0;
    SB_TRY(h2d(ctx, lv.u32[0], u, lv.M));
    SB_TRY(h2d(ctx, stage32(ctx, 1), rhs, lv.M));
    SB_TRY(sb_vcycle(ctx, level, smoother, pre, post, (const float *)stage32(ctx, 1), false));
    return d2h(ctx, u, lv.u32[lv.cur], lv.M);
}

// ---------------------------------------------------------------------------------------------
// block solve: k <= SB_BLOCK_MAX right-hand sides on one hierarchy, every operator streamed once for all of them.
// Column j gives what saena_b200_solve_pcg gives for right-hand side j: each column has its own alpha, beta, init_dot
// and stop test, and once it has stopped its u, r and p are left as they are (the PCG updates skip it) while the
// others go on; it still rides through the V-cycle and the SpMV, whose results it never reads.
// ---------------------------------------------------------------------------------------------
static int block_enter(saena_b200_ctx *ctx, int k) {
    if (k < 1 || k > SB_BLOCK_MAX) SB_FAIL("block call: k must be in 1..8");
    // column j is the single solve's bits: with the FP32 preconditioner that would be an FP32 block V-cycle
    if (ctx->precond_bits == 32) SB_FAIL("block call: not while the preconditioner precision is 32");
    if (ctx->nranks > 1) SB_FAIL("block call: one rank only (the halo exchange has no block form)");
    return sb_block_reserve(ctx, k);
}

#define SB_ENTER_BLOCK(k)                                                 \
    SB_ENTER();                                                           \
    SB_TRY(block_enter(ctx, k))

static int upload_active(saena_b200_ctx *ctx, int k) {
    SB_CUDA(cudaMemcpyAsync(ctx->blk_active, ctx->blk_active_host, sizeof(int) * k, cudaMemcpyHostToDevice,
                            ctx->stream));
    return 0;
}

static int pcg_block_device(saena_b200_ctx *ctx, int k, const double *rhs, double *u, int max_iter, double tol,
                            int smoother, int pre, int post, int *iters, double *hist, int hist_cap, int *hist_len) {
    DevLevel &l0 = ctx->levels[0];
    const int n = l0.M;
    const long long ld = n;
    if (ctx->levels.size() == 1) {
        // direct solver only (pcg_device :2507-2521): nothing to share, one column after the other
        for (int j = 0; j < k; ++j)
            SB_TRY(pcg_device(ctx, rhs + j * ld, u + j * ld, max_iter, tol, smoother, pre, post, iters + j,
                              hist ? hist + (long long)j * hist_cap : nullptr, hist_cap, hist_len + j));
        return 0;
    }
    double *r = ctx->blk_r, *p = ctx->blk_p, *h = ctx->blk_h;
    const double *sc = ctx->blk_scal_host;
    auto rr_of = [&](int j) { return sc[S_RR * SB_BLOCK_MAX + j]; };
    auto push = [&](int j, double v) { push_hist(v, hist ? hist + (long long)j * hist_cap : nullptr, hist_cap, hist_len[j]); };
    double thr[SB_BLOCK_MAX];
    int *active = ctx->blk_active_host;
    SB_TRY(sb_fill_zero(ctx, u, (size_t)k * n));
    SB_TRY(sb_negate_copy_block(ctx, n, k, rhs, r));
    SB_TRY(sb_dot_block(ctx, r, r, n, k, S_RR));
    SB_TRY(sb_read_block_scalars(ctx));
    for (int j = 0; j < k; ++j) {
        hist_len[j] = 0;
        iters[j] = max_iter;   // a column that never stops ends at max_iter (pcg_device :2673-2682)
        active[j] = 1;
        thr[j] = rr_of(j) * tol * tol;
        push(j, rr_of(j));
    }
    SB_TRY(upload_active(ctx, k));
    double *rho = nullptr;
    SB_TRY(sb_vcycle_block_from_zero(ctx, k, smoother, pre, post, r));
    rho = l0.bu[l0.bcur];
    if (n) SB_CUDA(cudaMemcpyAsync(p, rho, sizeof(double) * k * ld, cudaMemcpyDeviceToDevice, ctx->stream));
    SB_TRY(sb_dot_block(ctx, r, rho, n, k, S_RHO_RES));
    int n_active = k;
    for (int i = 0; i < max_iter && n_active; i++) {
        EpiArgs e{};
        e.out = h;
        SB_TRY(sb_apply_block(ctx, l0.A, k, p, EPI_PLAIN, e));
        SB_TRY(sb_dot_block(ctx, p, h, n, k, S_PDOTH));
        SB_TRY(sb_pcg_update_block(ctx, n, k, u, r, p, h));
        SB_TRY(sb_read_block_scalars(ctx));
        bool changed = false;
        for (int j = 0; j < k; ++j) {
            if (!active[j]) continue;
            push(j, rr_of(j));
            if (!(rr_of(j) >= thr[j])) {   // NaN also stops
                active[j] = 0;
                iters[j] = i + 1;
                --n_active;
                changed = true;
            }
        }
        if (!n_active) break;
        if (changed) SB_TRY(upload_active(ctx, k));
        SB_TRY(sb_vcycle_block_from_zero(ctx, k, smoother, pre, post, r));
        rho = l0.bu[l0.bcur];
        SB_TRY(sb_dot_block(ctx, r, rho, n, k, S_BETA_NUM));
        SB_TRY(sb_pcg_p_update_block(ctx, n, k, p, rho));
    }
    if (ctx->scale) SB_TRY(sb_scale_vector_block(ctx, n, k, u, l0.inv_sq_diag));
    return 0;
}

int saena_b200_solve_pcg_block_dev(saena_b200_ctx *ctx, int k, const double *rhs_dev, double *u_dev, int max_iter,
                                   double tol, int smoother, int pre, int post, int *iters, double *hist,
                                   int hist_cap, int *hist_len) {
    SB_ENTER_BLOCK(k);
    if (!iters || !hist_len || !rhs_dev || !u_dev) SB_FAIL("solve_pcg_block: null argument");
    SB_TRY(pcg_block_device(ctx, k, rhs_dev, u_dev, max_iter, tol, smoother, pre, post, iters, hist, hist_cap,
                            hist_len));
    SB_TRY(sb_sync_stream(ctx, ctx->stream));
    return sb_agree_fault(ctx);
}

int saena_b200_solve_pcg_block(saena_b200_ctx *ctx, int k, const double *rhs, double *u, int max_iter, double tol,
                               int smoother, int pre, int post, int *iters, double *hist, int hist_cap,
                               int *hist_len) {
    SB_ENTER_BLOCK(k);
    if (!iters || !hist_len || !rhs || !u) SB_FAIL("solve_pcg_block: null argument");
    const size_t n = (size_t)k * ctx->levels[0].M;
    SB_TRY(h2d(ctx, ctx->blk_rhs, rhs, n));
    SB_TRY(pcg_block_device(ctx, k, ctx->blk_rhs, ctx->blk_u, max_iter, tol, smoother, pre, post, iters, hist,
                            hist_cap, hist_len));
    SB_TRY(sb_agree_fault(ctx));
    return d2h(ctx, u, ctx->blk_u, n);
}

int saena_b200_matvec_block(saena_b200_ctx *ctx, int level, int kind, int k, const double *v, double *w) {
    SB_ENTER_BLOCK(k);
    DevOperator *op = get_op(ctx, level, kind);
    if (!op) SB_FAIL("matvec_block: no such operator");
    const size_t nx = (size_t)k * op->n_local_cols, nw = (size_t)k * op->M;
    SB_TRY(stage_buf(ctx, 0, nx));
    SB_TRY(stage_buf(ctx, 1, nw));
    SB_TRY(h2d(ctx, ctx->stage[0], v, nx));
    EpiArgs e{};
    e.out = ctx->stage[1];
    if (kind == SAENA_B200_KIND_A) SB_TRY(sb_apply_level_A_block(ctx, level, k, ctx->stage[0], EPI_PLAIN, e));
    else SB_TRY(sb_apply_block(ctx, *op, k, ctx->stage[0], EPI_PLAIN, e));
    return d2h(ctx, w, ctx->stage[1], nw);
}

int saena_b200_residual_block(saena_b200_ctx *ctx, int level, int k, const double *u, const double *rhs, double *res) {
    SB_ENTER_BLOCK(k);
    DevOperator *op = get_op(ctx, level, SAENA_B200_KIND_A);
    if (!op) SB_FAIL("residual_block: no such level");
    const size_t n = (size_t)k * op->M;
    for (int i = 0; i < 3; ++i) SB_TRY(stage_buf(ctx, i, n));
    SB_TRY(h2d(ctx, ctx->stage[0], u, n));
    SB_TRY(h2d(ctx, ctx->stage[1], rhs, n));
    EpiArgs e{};
    e.rhs = ctx->stage[1];
    e.out = ctx->stage[2];
    SB_TRY(sb_apply_level_A_block(ctx, level, k, ctx->stage[0], EPI_RESIDUAL, e));
    return d2h(ctx, res, ctx->stage[2], n);
}

int saena_b200_smooth_block(saena_b200_ctx *ctx, int level, int smoother, int iters, int k, double *u,
                            const double *rhs) {
    SB_ENTER_BLOCK(k);
    if (level < 0 || level >= (int)ctx->levels.size()) SB_FAIL("smooth_block: no such level");
    DevLevel &lv = ctx->levels[level];
    const size_t n = (size_t)k * lv.M;
    SB_TRY(stage_buf(ctx, 1, n));
    lv.bcur = 0;
    SB_TRY(h2d(ctx, lv.bu[0], u, n));
    SB_TRY(h2d(ctx, ctx->stage[1], rhs, n));
    SB_TRY(sb_smooth_block(ctx, level, k, smoother, iters, ctx->stage[1], false));
    return d2h(ctx, u, lv.bu[lv.bcur], n);
}

int saena_b200_vcycle_block(saena_b200_ctx *ctx, int level, int smoother, int pre, int post, int k, double *u,
                            const double *rhs) {
    SB_ENTER_BLOCK(k);
    if (level < 0 || level >= (int)ctx->levels.size()) SB_FAIL("vcycle_block: no such level");
    DevLevel &lv = ctx->levels[level];
    const size_t n = (size_t)k * lv.M;
    SB_TRY(stage_buf(ctx, 1, n));
    lv.bcur = 0;
    SB_TRY(h2d(ctx, lv.bu[0], u, n));
    SB_TRY(h2d(ctx, ctx->stage[1], rhs, n));
    SB_TRY(sb_vcycle_block(ctx, level, k, smoother, pre, post, ctx->stage[1], false));
    return d2h(ctx, u, lv.bu[lv.bcur], n);
}

// ---------------------------------------------------------------------------------------------
// measurement
// ---------------------------------------------------------------------------------------------
// median over the launches of a timing loop: robust against the odd launch that waits for a peer
static float median_of(std::vector<float> &t) {
    if (t.empty()) return 0.f;
    std::sort(t.begin(), t.end());
    const size_t n = t.size();
    return n % 2 ? t[n / 2] : 0.5f * (t[n / 2 - 1] + t[n / 2]);
}

static int flush_l2(saena_b200_ctx *ctx) {
    const size_t bytes = (size_t)256 << 20;  // > 126 MB L2
    if (!ctx->flush_buf) {
        SB_CUDA(cudaMalloc(&ctx->flush_buf, bytes));
        ctx->flush_bytes = bytes;
    }
    SB_CUDA(cudaMemsetAsync(ctx->flush_buf, 0, ctx->flush_bytes, ctx->stream));
    return 0;
}

int saena_b200_time_matvec(saena_b200_ctx *ctx, int level, int kind, int reps, int do_flush, float *ms_out) {
    SB_ENTER();
    DevOperator *op = get_op(ctx, level, kind);
    if (!op) SB_FAIL("time_matvec: no such operator");
    const bool f32 = ctx->precond_bits == 32;
    if (f32) SB_TRY(sb_f32_sync(ctx));
    SB_TRY(stage_buf(ctx, 0, op->n_local_cols));
    SB_TRY(stage_buf(ctx, 1, op->M));
    SB_CUDA(cudaMemsetAsync(ctx->stage[0], 0, sizeof(double) * op->n_local_cols, ctx->stream));
    EpiArgs e{};
    e.out = ctx->stage[1];
    EpiArgs32 e32{};
    e32.out = stage32(ctx, 1);
    std::vector<float> t;
    for (int it = 0; it < reps; ++it) {
        if (do_flush) SB_TRY(flush_l2(ctx));
        SB_CUDA(cudaEventRecord(ctx->ev_t0, ctx->stream));
        if (f32) SB_TRY(apply_kind(ctx, level, kind, (const float *)stage32(ctx, 0), EPI_PLAIN, e32));
        else SB_TRY(apply_kind(ctx, level, kind, (const double *)ctx->stage[0], EPI_PLAIN, e));
        SB_CUDA(cudaEventRecord(ctx->ev_t1, ctx->stream));
        SB_TRY(sb_sync_stream(ctx, ctx->stream));
        float ms = 0.f;
        SB_CUDA(cudaEventElapsedTime(&ms, ctx->ev_t0, ctx->ev_t1));
        t.push_back(ms);
    }
    *ms_out = median_of(t);
    return sb_check_fault(ctx);
}

// Picks, per operator, the faster of the two forms of the peer-memory exchange by measuring both on the
// uploaded hierarchy: the fused kernel (fused_halo.cu) wins where an application is latency-bound
// (coarse levels, many ranks), the separate launches (p2p_halo.cu: pack on the comm stream
// overlapping a plain interior kernel) can win on the big fine levels.  Collective: every rank
// times `reps` back-to-back applications of each operator both ways, the times are summed over
// the ranks (ncclAllReduce) and every rank takes the same decision from the same sums.
// Safety does not rest on that agreement: the two forms speak one hand-shake on the same counters and landing
// buffers (halo_sync.cuh), so a rank whose operator cannot take the fused kernel (64-bit row offsets, a forced
// streaming mapping) simply runs the separate launches in both timing loops while its neighbours run what they like.
// Every rank holds every level (empty where it owns no row), so all ranks walk the same (level, operator) list and
// join the same all-reduces.
int saena_b200_autotune_halo(saena_b200_ctx *ctx, int reps) {
    SB_ENTER();
    if (ctx->nranks == 1 || !ctx->p2p_ready) return 0;
    if (reps < 1) reps = 10;
    sb_invalidate_graphs(ctx);
    const size_t n_walk = ctx->levels.size();
    for (size_t l = 0; l < n_walk; ++l) {
        DevOperator *ops[3] = {&ctx->levels[l].A, &ctx->levels[l].P, &ctx->levels[l].R};
        for (DevOperator *op : ops) {
            double ms2[2] = {0.0, 0.0};
            const bool mine = op->present && op->p2p && op->hs.epoch && (!op->sends.empty() || !op->recvs.empty());
            if (mine) {
                SB_TRY(stage_buf(ctx, 0, op->n_local_cols));
                SB_TRY(stage_buf(ctx, 1, op->M));
                SB_CUDA(cudaMemsetAsync(ctx->stage[0], 0, sizeof(double) * op->n_local_cols, ctx->stream));
                EpiArgs e{};
                e.out = ctx->stage[1];
                for (int mode = 0; mode < 2; ++mode) {
                    op->fused = mode == 0;   // not eligible: sb_apply takes the separate launches, same protocol
                    for (int it = -2; it < reps; ++it) {
                        if (it == 0) SB_CUDA(cudaEventRecord(ctx->ev_t0, ctx->stream));
                        SB_TRY(sb_apply(ctx, *op, ctx->stage[0], EPI_PLAIN, e));
                    }
                    SB_CUDA(cudaEventRecord(ctx->ev_t1, ctx->stream));
                    SB_TRY(sb_sync_stream(ctx, ctx->stream));
                    SB_TRY(sb_sync_stream(ctx, ctx->comm_stream));
                    float ms = 0.f;
                    SB_CUDA(cudaEventElapsedTime(&ms, ctx->ev_t0, ctx->ev_t1));
                    ms2[mode] = ms / reps;
                }
            }
            if (op->present) { op->tune_ms[0] = (float)ms2[0]; op->tune_ms[1] = (float)ms2[1]; }
            // same decision on every rank: sum over ranks (ranks without a halo on this operator add 0)
            SB_CUDA(cudaMemcpyAsync(ctx->scalars + S_TMP, ms2, sizeof(ms2), cudaMemcpyHostToDevice, ctx->stream));
            SB_TRY(sb_allreduce_sum(ctx, ctx->scalars + S_TMP, 2, ctx->stream));
            SB_TRY(sb_read_scalars(ctx));
            const double f = ctx->scalars_host[S_TMP], u = ctx->scalars_host[S_TMP + 1];
            if (op->present && op->p2p && op->hs.epoch) op->fused = f <= u;
        }
    }
    return sb_agree_fault(ctx);
}

}  // extern "C"

// median ms of `reps` calls of apply() (two untimed first), each bracketed by CUDA events
template <typename F>
static int time_median(saena_b200_ctx *ctx, int reps, bool flush, F apply, float *ms_out) {
    std::vector<float> t;
    for (int it = -2; it < reps; ++it) {
        if (flush) SB_TRY(flush_l2(ctx));
        SB_CUDA(cudaEventRecord(ctx->ev_t0, ctx->stream));
        SB_TRY(apply());
        SB_CUDA(cudaEventRecord(ctx->ev_t1, ctx->stream));
        SB_TRY(sb_sync_stream(ctx, ctx->stream));
        float ms = 0.f;
        SB_CUDA(cudaEventElapsedTime(&ms, ctx->ev_t0, ctx->ev_t1));
        if (it >= 0) t.push_back(ms);
    }
    *ms_out = median_of(t);
    return 0;
}

extern "C" {

static int time_apply_median(saena_b200_ctx *ctx, DevOperator *op, int reps, bool flush, float *ms_out) {
    EpiArgs e{};
    e.out = ctx->stage[1];
    return time_median(ctx, reps, flush, [&]() { return sb_apply(ctx, *op, ctx->stage[0], EPI_PLAIN, e); }, ms_out);
}

// ---------------------------------------------------------------------------------------------
// Level route (sb_apply_level_A): level l's operator applied as R_{l-1} A_{l-1} P_{l-1}.
// ---------------------------------------------------------------------------------------------
// nullptr when level l may take the route, else why not.  One rank only: on several ranks each of the three operators
// would need its own halo exchange.  The scaled path and the repartitioned levels store an A_l that is not R A P of the
// operators next to it; a dense level rounds its input through float.
static const char *route_refusal(const saena_b200_ctx *ctx, int l) {
    if (ctx->nranks != 1) return "one rank only";
    if (ctx->scale) return "not on a scaled hierarchy";
    if (l < 1 || l >= (int)ctx->levels.size()) return "no level above this one";
    const DevLevel &lv = ctx->levels[l], &fl = ctx->levels[l - 1];
    if (!fl.repart.identity()) return "the level above repartitions its coarse vector";
    for (const DevOperator *op : {&lv.A, &fl.A, &fl.P, &fl.R}) {
        if (!op->present) return "an operator of the route is missing";
        if (!op->sends.empty() || !op->recvs.empty() || op->nnz_remote > 0 || op->merged) return "an operator has a halo";
        if (op->use_dense) return "an operator is on the dense path";
    }
    return nullptr;
}

// the intermediates are kept only while some level is on the route
static void route_release_if_unused(saena_b200_ctx *ctx) {
    for (const DevLevel &lv : ctx->levels)
        if (lv.route) return;
    route_free(ctx);
}

// Largest ||route x - A_l x|| / ||A_l x|| over two seeded random x.  The difference comes out of the route's last
// SpMV directly (residual epilogue against the stored product), so no digits are lost to cancellation.
static const double ROUTE_PROBE_TOL = 1e-12;

static int route_probe(saena_b200_ctx *ctx, int l, double *rel_out) {
    DevLevel &lv = ctx->levels[l];
    const int n = lv.M;
    for (int i = 0; i < 3; ++i) SB_TRY(stage_buf(ctx, i, n));
    SB_TRY(route_alloc(ctx, ctx->levels[l - 1].M));
    const bool was = lv.route;
    double worst = 0.0;
    for (unsigned long long seed = 1; seed <= 2; ++seed) {
        SB_TRY(sb_fill_random(ctx, n, 0, 0x5EEDull + seed, ctx->stage[0]));
        EpiArgs e{};
        e.out = ctx->stage[1];
        lv.route = false;
        SB_TRY(sb_apply_level_A(ctx, l, ctx->stage[0], EPI_PLAIN, e));   // stored A_l x
        e.rhs = ctx->stage[1];
        e.out = ctx->stage[2];
        lv.route = true;
        const int rc = sb_apply_level_A(ctx, l, ctx->stage[0], EPI_RESIDUAL, e);   // route x - A_l x
        lv.route = was;
        SB_TRY(rc);
        SB_TRY(sb_dot(ctx, ctx->stage[2], ctx->stage[2], n, S_TMP));
        SB_TRY(sb_dot(ctx, ctx->stage[1], ctx->stage[1], n, S_TMP + 1));
        SB_TRY(sb_read_scalars(ctx));
        const double num = ctx->scalars_host[S_TMP], den = ctx->scalars_host[S_TMP + 1];
        const double r = den > 0.0 ? sqrt(num / den) : (num > 0.0 ? INFINITY : 0.0);
        if (!(r <= worst)) worst = r;   // NaN stays
    }
    *rel_out = worst;
    return 0;
}

int saena_b200_set_level_route(saena_b200_ctx *ctx, int level, int on) {
    SB_ENTER();
    if (level < 0 || level >= (int)ctx->levels.size()) SB_FAIL("set_level_route: no such level");
    DevLevel &lv = ctx->levels[level];
    sb_invalidate_graphs(ctx);
    if (!on) {
        lv.route = false;
        route_release_if_unused(ctx);
        return 0;
    }
    if (const char *why = route_refusal(ctx, level)) SB_FAIL(std::string("set_level_route: ") + why);
    double rel = 0.0;
    const int rc = route_probe(ctx, level, &rel);
    if (rc || !(rel <= ROUTE_PROBE_TOL)) {
        route_release_if_unused(ctx);
        if (rc) return rc;
        SB_FAIL("set_level_route: R A P of the level above differs from the stored operator by " + std::to_string(rel) +
                " relative (more than 1e-12)");
    }
    lv.route = true;
    return 0;
}

int saena_b200_get_level_route(const saena_b200_ctx *ctx, int level, float *ms_stored, float *ms_route) {
    if (!ctx || level < 0 || level >= (int)ctx->levels.size()) return -1;
    const DevLevel &lv = ctx->levels[level];
    if (ms_stored) *ms_stored = lv.route_ms[0];
    if (ms_route) *ms_route = lv.route_ms[1];
    return lv.route ? 1 : 0;
}

// Setup-time choice of the route, after the mappings are settled: for every level it may take, the stored operator and
// the route are each timed as the V-cycle's most frequent application, a Chebyshev sweep after the first, and the route
// is kept where it is faster by more than min_gain.  Tried only where the three operators together stream fewer bytes
// than the stored one and pass the probe check.  The coarsest level is left alone: the V-cycle never applies its A.
static int autotune_route(saena_b200_ctx *ctx, int reps, double min_gain) {
    for (int l = 1; l + 1 < (int)ctx->levels.size(); ++l) {
        DevLevel &lv = ctx->levels[l], &fl = ctx->levels[l - 1];
        lv.route = false;
        lv.route_ms[0] = lv.route_ms[1] = 0.f;
        if (route_refusal(ctx, l) || lv.M == 0) continue;
        const int64_t stored = sb_operator_bytes(lv.A);
        if (sb_operator_bytes(fl.P) + sb_operator_bytes(fl.A) + sb_operator_bytes(fl.R) >= stored) continue;
        double rel = 0.0;
        SB_TRY(route_probe(ctx, l, &rel));
        if (!(rel <= ROUTE_PROBE_TOL)) continue;
        // stage[0]: iterate and rhs (zeros), stage[1]: new iterate, stage[2]: direction (in place, as in the solve)
        SB_CUDA(cudaMemsetAsync(ctx->stage[0], 0, sizeof(double) * lv.M, ctx->stream));
        SB_CUDA(cudaMemsetAsync(ctx->stage[2], 0, sizeof(double) * lv.M, ctx->stream));
        EpiArgs e{};
        e.rhs = ctx->stage[0];
        e.inv_diag = lv.inv_diag;
        e.d_in = e.d_out = ctx->stage[2];
        e.u_in = ctx->stage[0];
        e.out = ctx->stage[1];
        e.c1 = 0.5;
        e.c2 = 0.5;
        const bool flush = stored < (int64_t)300e6;
        float ms[2] = {0.f, 0.f};
        for (int r = 0; r < 2; ++r) {
            lv.route = r == 1;
            SB_TRY(time_median(ctx, reps, flush, [&]() { return sb_apply_level_A(ctx, l, ctx->stage[0], EPI_CHEB_NEXT, e); },
                               &ms[r]));
        }
        lv.route_ms[0] = ms[0];
        lv.route_ms[1] = ms[1];
        lv.route = ms[1] < (1.0 - min_gain) * ms[0];
    }
    route_release_if_unused(ctx);
    return 0;
}

// ---------------------------------------------------------------------------------------------
// Setup-time choice of every operator's row mapping BY MEASUREMENT (north_star: "warp-per-row or row-block mapping
// chosen per level by nnz/row"): sb_choose_mapping's nnz/row rule gives the starting point, this walks the
// neighbouring mappings -- 1/8 .. 8x the threads per row, and the sorted sliced layout (101) where short irregular
// rows run on a sub-warp mapping -- times `reps` applications of each with the library's own launcher and keeps the
// fastest when it wins by more than min_gain.  Round 2 measurement behind it (profiles/r02_mapping_autotune.md): the
// rule was up to 27 % off on the transfer operators of level 2 and 12 % on level 3's A (256 -> 64 threads per row).
// Collective on several ranks: every rank walks the same operators and the same candidates (derived from the
// all-reduced maximum of the ranks' starting points), every timed application of an operator with a halo is an
// exchange all ranks take part in, and the decision is taken on the slowest rank's median time (all-reduce MAX) --
// one mapping per operator on all ranks.  Sliced operators (mapping 100) keep a sliced layout: where the rule picks it,
// it measured fastest on every shape tried (profiles/r01_mapping_sweep.md); on one rank they are timed against the
// sorted sliced layout (101).
// changed_out (optional): number of operators whose mapping changed on this rank.  On one rank the level route is
// chosen afterwards, on the settled mappings (autotune_route).
// ---------------------------------------------------------------------------------------------
int saena_b200_autotune_mapping(saena_b200_ctx *ctx, int reps, double min_gain, int *changed_out) {
    SB_ENTER();
    if (reps < 3) reps = 10;
    if (!(min_gain >= 0.0)) min_gain = 0.03;
    if (!ctx->tune_dev) SB_CUDA(cudaMalloc((void **)&ctx->tune_dev, sizeof(double) * 32));
    sb_invalidate_graphs(ctx);
    int changed = 0;
    const bool multi = ctx->nranks > 1 && !ctx->detached;
    for (size_t l = 0; l < ctx->levels.size(); ++l) {
        DevOperator *ops[3] = {&ctx->levels[l].A, &ctx->levels[l].P, &ctx->levels[l].R};
        for (int kind = 0; kind < 3; ++kind) {
            DevOperator *op = ops[kind];
            // ---- what this rank holds
            const bool mine = op->present && op->M > 0 && op->nnz_local + op->nnz_remote > 0;
            const int cur = mine ? op->mapping : 0;
            const bool has_halo = mine && (!op->sends.empty() || !op->recvs.empty() || op->nnz_remote > 0 || op->merged);
            // ---- one rank, sliced, no halo: the same layout over rows sorted by length (101) against it.  One lane
            //      sums a row in column order in both (same result, bit for bit); the sorted layout streams less
            //      padding where the rows of a 32-row slice differ in length (the 267-entry rows of level 2 of the
            //      256^3 hierarchy), at the price of a permutation and a pass through shared memory.  An eligible symmetric
            //      operator (the rule put it on 103) is timed on the symmetric diagonals against both.
            if (!multi && mine && (cur == SB_MAPPING_SELL || cur == SB_MAPPING_SYMDIAG) && !op->sell_only && !has_halo) {
                SB_TRY(stage_buf(ctx, 0, op->n_local_cols));
                SB_TRY(stage_buf(ctx, 1, op->M));
                SB_CUDA(cudaMemsetAsync(ctx->stage[0], 0, sizeof(double) * op->n_local_cols, ctx->stream));
                const bool flush = sb_operator_bytes(*op) < (int64_t)300e6;
                // the symmetric diagonals (103) where the operator is eligible; the rule's choice is the base
                std::vector<int> cands = {SB_MAPPING_SELL, SB_MAPPING_SELLP};
                if (op->sdiag_n > 0) cands.push_back(SB_MAPPING_SYMDIAG);
                std::vector<float> t(cands.size(), 0.f);
                size_t best = 0, base = 0;
                for (size_t k = 0; k < cands.size(); ++k) {
                    op->forced_mapping = cands[k];
                    SB_TRY(sb_prepare_operator(ctx, *op));
                    SB_TRY(time_apply_median(ctx, op, reps, flush, &t[k]));
                    if (cands[k] == cur) base = k;
                    if (t[k] < t[best]) best = k;
                }
                if (!(t[best] < (1.0 - min_gain) * t[base])) best = base;
                op->forced_mapping = cands[best];
                SB_TRY(sb_prepare_operator(ctx, *op));
                SB_CUDA(cudaStreamSynchronize(ctx->stream));
                sb_drop_unused_layouts(*op);
                if (op->mapping != cur) ++changed;
                continue;
            }
            // ---- agree: [largest threads-per-row starting point, somebody is sliced / streaming / pinned]
            double agree[2] = {(cur >= 1 && cur <= 256) ? (double)cur : 0.0,
                               (mine && (cur <= 0 || cur >= SB_MAPPING_SELL || op->sell_only)) ? 1.0 : 0.0};
            if (multi) {
                SB_CUDA(cudaMemcpyAsync(ctx->tune_dev, agree, sizeof(agree), cudaMemcpyHostToDevice, ctx->stream));
                SB_TRY(sb_allreduce_max(ctx, ctx->tune_dev, 2, ctx->stream));
                SB_CUDA(cudaMemcpyAsync(agree, ctx->tune_dev, sizeof(agree), cudaMemcpyDeviceToHost, ctx->stream));
                SB_TRY(sb_sync_stream(ctx, ctx->stream));
            }
            const int start = (int)agree[0];
            if (start == 0 || agree[1] != 0.0) continue;   // nobody holds it, or a mapping this walk leaves alone
            // ---- candidates, the same list on every rank
            std::vector<int> cands;
            for (int c = 1; c <= 256; c *= 2)
                if (c * 8 >= start && c <= start * 8) cands.push_back(c);
            if (!multi && mine && !has_halo && start < 32 && op->M >= 150000) cands.push_back(SB_MAPPING_SELLP);
            std::vector<double> ms(32, 0.0);
            if (mine) {
                SB_TRY(stage_buf(ctx, 0, op->n_local_cols));
                SB_TRY(stage_buf(ctx, 1, op->M));
                SB_CUDA(cudaMemsetAsync(ctx->stage[0], 0, sizeof(double) * op->n_local_cols, ctx->stream));
            }
            const bool flush = mine && sb_operator_bytes(*op) < (int64_t)300e6;
            for (size_t k = 0; k < cands.size(); ++k) {
                if (!mine) continue;   // no row, no halo: nothing of this operator to run, only the agreement below
                op->forced_mapping = cands[k];
                SB_TRY(sb_prepare_operator(ctx, *op));
                float t = 0.f;
                SB_TRY(time_apply_median(ctx, op, reps, flush, &t));
                ms[k] = t;
            }
            if (multi) {
                SB_CUDA(cudaMemcpyAsync(ctx->tune_dev, ms.data(), sizeof(double) * 32, cudaMemcpyHostToDevice, ctx->stream));
                SB_TRY(sb_allreduce_max(ctx, ctx->tune_dev, 32, ctx->stream));
                SB_CUDA(cudaMemcpyAsync(ms.data(), ctx->tune_dev, sizeof(double) * 32, cudaMemcpyDeviceToHost, ctx->stream));
                SB_TRY(sb_sync_stream(ctx, ctx->stream));
            }
            // ---- decision: the fastest; the starting point unless it is beaten by more than min_gain
            size_t best = 0, base = 0;
            for (size_t k = 0; k < cands.size(); ++k) {
                if (cands[k] == start) base = k;
                if (ms[k] < ms[best]) best = k;
            }
            if (!(ms[best] < (1.0 - min_gain) * ms[base])) best = base;
            if (mine) {
                op->forced_mapping = cands[best];
                SB_TRY(sb_prepare_operator(ctx, *op));
                SB_CUDA(cudaStreamSynchronize(ctx->stream));
                sb_drop_unused_layouts(*op);
                if (cands[best] != cur) ++changed;
            }
        }
    }
    if (changed_out) *changed_out = changed;
    if (multi) return sb_agree_fault(ctx);
    return ctx->nranks == 1 ? autotune_route(ctx, reps, min_gain) : 0;
}

// 1: fused kernel, 0: separate launches / NCCL, -1: no such operator; ms[2] = this rank's autotune timings
int saena_b200_halo_choice(const saena_b200_ctx *ctx, int level, int kind, float *ms_fused, float *ms_unfused) {
    if (!ctx || level < 0 || level >= (int)ctx->levels.size()) return -1;
    const DevOperator &op = ctx->levels[level].op(kind);
    if (!op.present) return -1;
    if (ms_fused) *ms_fused = op.tune_ms[0];
    if (ms_unfused) *ms_unfused = op.tune_ms[1];
    return op.fused && sb_fused_eligible(op) ? 1 : 0;
}

// SURVEY 8f #1: saena_object::find_eig on the device (csrc/lanczos.cu).  start: optional host start
// vector (this rank's rows), else a seeded generator on the global row index.  store != 0 makes the
// result the level's Chebyshev bound (what find_eig writes into eig_max_of_invdiagXA).
int saena_b200_find_eig(saena_b200_ctx *ctx, int level, int max_iter, const double *start, uint64_t seed, int store,
                        double *eig_out, int *iters_out) {
    SB_ENTER();
    if (level < 0 || level >= (int)ctx->levels.size() || !eig_out) SB_FAIL("find_eig: no such level");
    DevLevel &lv = ctx->levels[level];
    const double *start_dev = nullptr;
    if (start) {
        SB_TRY(stage_buf(ctx, 2, lv.M));
        SB_TRY(h2d(ctx, ctx->stage[2], start, lv.M));
        start_dev = ctx->stage[2];
    }
    SB_TRY(sb_find_eig(ctx, level, max_iter, start_dev, (unsigned long long)seed, eig_out, iters_out));
    if (store) {
        lv.eig_max = *eig_out;
        sb_invalidate_graphs(ctx);  // the captured V-cycle carries the old Chebyshev constants
    }
    return 0;
}

// Next to find_eig: new values for level 0's A, every coarse level recomputed on its stored pattern (refresh.cu).
// The host variant stages the values in stage[3], which no other entry point uses.
int saena_b200_update_values(saena_b200_ctx *ctx, const double *val_local, int64_t nnz_local, int max_eig_iter,
                             uint64_t seed, double *dropped_out, int dropped_cap) {
    SB_ENTER();
    if (nnz_local < 0 || (nnz_local && !val_local)) SB_FAIL("update_values: no values");
    SB_TRY(stage_buf(ctx, 3, (size_t)nnz_local));   // the caller's array holds nnz_local values; checked next
    SB_TRY(h2d(ctx, ctx->stage[3], val_local, (size_t)nnz_local));
    return sb_update_values(ctx, ctx->stage[3], nnz_local, max_eig_iter, (unsigned long long)seed, dropped_out,
                            dropped_cap);
}

int saena_b200_update_values_dev(saena_b200_ctx *ctx, const double *val_local_dev, int64_t nnz_local, int max_eig_iter,
                                 uint64_t seed, double *dropped_out, int dropped_cap) {
    SB_ENTER();
    if (nnz_local < 0 || (nnz_local && !val_local_dev)) SB_FAIL("update_values: no values");
    return sb_update_values(ctx, val_local_dev, nnz_local, max_eig_iter, (unsigned long long)seed, dropped_out,
                            dropped_cap);
}

int saena_b200_update_values_times(const saena_b200_ctx *ctx, double *ms_out, int cap) {
    if (!ctx || !ms_out) return 1;
    for (int i = 0; i < cap && i < 5; ++i) ms_out[i] = ctx->update_ms[i];
    return 0;
}

// compute side only (apply_mode 1: no pack, no flags, no exchange; ghost values as they lie) of one
// operator, through the fused kernel (fused != 0) or the separate interior + boundary kernels.  The one
// timing hook a detached context (saena_b200_init_detached) supports; also valid on a live one.
int saena_b200_time_matvec_compute_only(saena_b200_ctx *ctx, int level, int kind, int fused, int reps, int do_flush,
                                        float *ms_out) {
    SB_ENTER();
    DevOperator *op = get_op(ctx, level, kind);
    if (!op) SB_FAIL("time_matvec_compute_only: no such operator");
    const bool was = op->fused, was_p2p = op->p2p;
    op->fused = fused != 0;
    if (fused && ctx->detached) op->p2p = true;   // compute roles only: the hand-shake state is never touched
    ctx->apply_mode = 1;
    int rc = saena_b200_time_matvec(ctx, level, kind, 3, 0, ms_out);
    if (!rc) rc = saena_b200_time_matvec(ctx, level, kind, reps, do_flush, ms_out);
    ctx->apply_mode = 0;
    op->fused = was;
    op->p2p = was_p2p;
    return rc;
}

// halo overlap of one operator: full application, local kernels alone, pack + exchange alone
int saena_b200_time_matvec_parts(saena_b200_ctx *ctx, int level, int kind, int reps, float *full_ms,
                                 float *local_ms, float *halo_ms) {
    SB_ENTER();
    float *out[3] = {full_ms, local_ms, halo_ms};
    for (int mode = 0; mode < 3; ++mode) {
        ctx->apply_mode = mode;
        int rc = saena_b200_time_matvec(ctx, level, kind, 3, 0, out[mode]);  // warm-up
        if (!rc) rc = saena_b200_time_matvec(ctx, level, kind, reps, 0, out[mode]);
        ctx->apply_mode = 0;
        if (rc) return rc;
    }
    return 0;
}

int saena_b200_time_smooth_sweep(saena_b200_ctx *ctx, int level, int smoother, int reps, int do_flush,
                                 float *ms_out) {
    SB_ENTER();
    if (level < 0 || level >= (int)ctx->levels.size()) SB_FAIL("time_smooth_sweep: no such level");
    DevLevel &lv = ctx->levels[level];
    const bool f32 = ctx->precond_bits == 32;
    if (f32) SB_TRY(sb_f32_sync(ctx));
    SB_TRY(stage_buf(ctx, 1, lv.M));
    SB_CUDA(cudaMemsetAsync(ctx->stage[1], 0, sizeof(double) * lv.M, ctx->stream));
    std::vector<float> t;
    for (int it = 0; it < reps; ++it) {
        if (do_flush) SB_TRY(flush_l2(ctx));
        SB_CUDA(cudaEventRecord(ctx->ev_t0, ctx->stream));
        if (f32) SB_TRY(sb_smooth(ctx, level, smoother, 1, (const float *)stage32(ctx, 1), false));
        else SB_TRY(sb_smooth(ctx, level, smoother, 1, (const double *)ctx->stage[1], false));
        SB_CUDA(cudaEventRecord(ctx->ev_t1, ctx->stream));
        SB_TRY(sb_sync_stream(ctx, ctx->stream));
        float ms = 0.f;
        SB_CUDA(cudaEventElapsedTime(&ms, ctx->ev_t0, ctx->ev_t1));
        t.push_back(ms);
    }
    *ms_out = median_of(t);
    return 0;
}

// `reps` back-to-back V-cycles entered at `level` with a zero iterate (eager launches, collective),
// CUDA events on the compute stream; ms per V-cycle.  T(level) - T(level+1) is what one level costs
// inside the flow of a solve (bench.py's per-level share table).
int saena_b200_time_vcycle(saena_b200_ctx *ctx, int level, int smoother, int pre, int post, int reps, float *ms_out) {
    SB_ENTER();
    if (level < 0 || level >= (int)ctx->levels.size() || reps < 1) SB_FAIL("time_vcycle: no such level");
    DevLevel &lv = ctx->levels[level];
    const bool f32 = ctx->precond_bits == 32;
    if (f32) SB_TRY(sb_f32_sync(ctx));
    const double *rhs = level == 0 ? ctx->pcg_r : lv.rhs;
    for (int it = -1; it < reps; ++it) {   // one untimed pass first
        if (it == 0) SB_CUDA(cudaEventRecord(ctx->ev_t0, ctx->stream));
        for (size_t l = level; l < ctx->levels.size(); ++l) ctx->levels[l].cur = 0;
        if (f32) SB_TRY(sb_vcycle(ctx, level, smoother, pre, post, (const float *)lv.rhs32, true));
        else SB_TRY(sb_vcycle(ctx, level, smoother, pre, post, rhs, true));
    }
    SB_CUDA(cudaEventRecord(ctx->ev_t1, ctx->stream));
    SB_TRY(sb_sync_stream(ctx, ctx->stream));
    SB_TRY(sb_sync_stream(ctx, ctx->comm_stream));
    float ms = 0.f;
    SB_CUDA(cudaEventElapsedTime(&ms, ctx->ev_t0, ctx->ev_t1));
    *ms_out = ms / reps;
    return 0;
}

int saena_b200_timer_start(saena_b200_ctx *ctx) {
    if (!ctx) return 1;
    SB_CUDA(cudaSetDevice(ctx->device));
    SB_TRY(sb_sync_stream(ctx, ctx->stream));
    SB_CUDA(cudaEventRecord(ctx->ev_t0, ctx->stream));
    return 0;
}

int saena_b200_timer_stop(saena_b200_ctx *ctx, float *ms_out) {
    if (!ctx) return 1;
    SB_CUDA(cudaSetDevice(ctx->device));
    SB_CUDA(cudaEventRecord(ctx->ev_t1, ctx->stream));
    SB_TRY(sb_sync_stream(ctx, ctx->stream));
    SB_CUDA(cudaEventElapsedTime(ms_out, ctx->ev_t0, ctx->ev_t1));
    return 0;
}

int64_t saena_b200_launch_count(const saena_b200_ctx *ctx) { return ctx ? ctx->launches : 0; }

int saena_b200_set_mapping(saena_b200_ctx *ctx, int level, int kind, int mapping) {
    if (!ctx) return 1;
    SB_CUDA(cudaSetDevice(ctx->device));
    DevOperator *op = get_op(ctx, level, kind);
    if (!op) SB_FAIL("set_mapping: no such operator");
    if (op->sell_only && mapping != 0 && mapping != SB_MAPPING_SELL)
        SB_FAIL("set_mapping: this operator kept only its sliced copy");
    op->forced_mapping = mapping;
    sb_invalidate_graphs(ctx);
    return sb_prepare_operator(ctx, *op);
}

// records the mapping only; the next finalize prepares the operator with it (no layout is built
// for a mapping that is about to be replaced -- matters when the operator fills half the HBM)
int saena_b200_set_mapping_deferred(saena_b200_ctx *ctx, int level, int kind, int mapping) {
    if (!ctx) return 1;
    DevOperator *op = get_op(ctx, level, kind);
    if (!op) SB_FAIL("set_mapping_deferred: no such operator");
    op->forced_mapping = mapping;
    ctx->finalized = false;
    return 0;
}

int saena_b200_set_operator_dense(saena_b200_ctx *ctx, int level, int kind, int use_dense) {
    if (!ctx) return 1;
    SB_CUDA(cudaSetDevice(ctx->device));
    DevOperator *op = get_op(ctx, level, kind);
    if (!op) SB_FAIL("set_operator_dense: no such operator");
    if (kind != SAENA_B200_KIND_A) SB_FAIL("set_operator_dense: only A operators have a dense form (saena_matrix::use_dense)");
    op->use_dense = use_dense != 0;
    if (op->use_dense && !op->use_double && !op->x_round)
        SB_CUDA(cudaMalloc((void **)&op->x_round, sizeof(double) * (size_t)std::max(op->n_local_cols, 1)));
    sb_invalidate_graphs(ctx);
    return 0;
}

int saena_b200_set_coarsest_solver(saena_b200_ctx *ctx, int use_cg) {
    if (!ctx) return 1;
    if (ctx->coarsest_cg != (use_cg != 0)) {
        ctx->coarsest_cg = use_cg != 0;
        sb_invalidate_graphs(ctx);
    }
    return 0;
}

int saena_b200_set_graphs(saena_b200_ctx *ctx, int on) {
    if (!ctx) return 1;
    ctx->use_graphs = on != 0;
    if (!on) sb_invalidate_graphs(ctx);
    return 0;
}

int64_t saena_b200_graph_replays(const saena_b200_ctx *ctx) { return ctx ? ctx->graph_replays : 0; }

int saena_b200_sellp_layout(int M, const int64_t *rowptr, int32_t *perm, long long *slice_ptr) {
    if (M < 0 || !rowptr || !perm || !slice_ptr) return 1;
    sb_sellp_layout(M, rowptr, perm, slice_ptr);
    return 0;
}

int saena_b200_symdiag_plan(int M, int n_offsets, const int32_t *offsets, int64_t nnz, int64_t padded_est,
                            int32_t *stored) {
    if (n_offsets < 0 || (n_offsets && !offsets) || !stored) return -1;
    return sb_symdiag_plan(M, n_offsets, offsets, nnz, padded_est, stored);
}

int saena_b200_get_mapping(const saena_b200_ctx *ctx, int level, int kind) {
    if (!ctx || level < 0 || level >= (int)ctx->levels.size()) return 0;
    const DevOperator &op = ctx->levels[level].op(kind);
    return op.present ? op.mapping : 0;
}

int64_t saena_b200_operator_bytes(const saena_b200_ctx *ctx, int level, int kind) {
    if (!ctx || level < 0 || level >= (int)ctx->levels.size()) return -1;
    const DevOperator &op = ctx->levels[level].op(kind);
    if (!op.present) return -1;
    const int vb = ctx->precond_bits == 32 ? 4 : 8;   // what the V-cycle streams
    return kind == SAENA_B200_KIND_A ? sb_level_A_bytes(ctx, level, vb) : sb_operator_bytes(op, vb);
}

}  // extern "C"

// After the operators' values changed (saena_b200_update_values): a level stays on the route only while R A P of the
// level above still matches its stored operator to the probe's tolerance.
int sb_recheck_routes(saena_b200_ctx *ctx) {
    for (int l = 1; l < (int)ctx->levels.size(); ++l) {
        DevLevel &lv = ctx->levels[l];
        if (!lv.route) continue;
        double rel = 0.0;
        SB_TRY(route_probe(ctx, l, &rel));
        if (!(rel <= ROUTE_PROBE_TOL)) lv.route = false;
    }
    route_release_if_unused(ctx);
    return 0;
}
