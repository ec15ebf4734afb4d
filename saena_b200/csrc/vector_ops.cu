// vector_ops.cu -- streaming vector kernels of the Krylov loop and the coarsest-level apply.
//
//   dotProduct            /root/reference/include/aux_functions.h:116-123
//   PCG axpys             /root/reference/src/saena_object_solve.cpp:2593-2596, :2665-2667
//   coarsest direct solve /root/reference/src/saena_object_solve.cpp:793-958 (SuperLU_DIST pdgssvx)
//
// Reductions are deterministic: every CTA writes one partial, the last CTA to finish (atomic
// ticket) adds the partials in index order.  The scalars of the Krylov recurrences live in
// device memory (ctx->scalars) so alpha/beta never round-trip through the host.
//
// Block forms (saena_b200_solve_pcg_block): the same kernels on a grid with one row of CTAs per column (grid.y =
// column j, vectors at + j * ld); each column has its own partials, counter and scalars (stride sstride) and so the
// single call's CTA count, reduction tree and bits.  A single call is the grid with one row.
#include <nvtx3/nvToolsExt.h>
#include <stdio.h>

#include "common.h"

static inline int red_blocks(const saena_b200_ctx *ctx, int n) {
    int b = (n + 1023) / 1024;  // 256 threads x 4 elements
    const int cap = ctx->sm_count * 8 < RED_MAX_BLOCKS ? ctx->sm_count * 8 : RED_MAX_BLOCKS;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return b;
}

__device__ __forceinline__ double block_sum_256(double v, double *s_w) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x < 32) {
        t = threadIdx.x < (blockDim.x >> 5) ? s_w[threadIdx.x] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    }
    return t;  // valid in thread 0
}

// last-CTA finalisation: partials[0..gridDim) summed in index order by one warp
__device__ __forceinline__ void finalize_sum(double block_total, double *partials, unsigned int *counter,
                                             double *out) {
    __shared__ bool s_last;
    if (threadIdx.x == 0) {
        partials[blockIdx.x] = block_total;
        __threadfence();
        const unsigned int ticket = atomicAdd(counter, 1u);
        s_last = (ticket == gridDim.x - 1);
    }
    __syncthreads();
    if (s_last && threadIdx.x < 32) {
        double t = 0.0;
        for (unsigned int i = threadIdx.x; i < gridDim.x; i += 32) t += __ldcg(partials + i);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        if (threadIdx.x == 0) {
            *out = t;
            *counter = 0u;
        }
    }
}

__global__ void __launch_bounds__(256)
dot_kernel(int n, long long ld, const double *__restrict__ a, const double *__restrict__ b, double *partials,
           unsigned int *counter, double *out) {
    __shared__ double s_w[8];
    const long long o = blockIdx.y * ld;
    a += o;
    b += o;
    partials += blockIdx.y * RED_MAX_BLOCKS;
    counter += blockIdx.y;
    out += blockIdx.y;
    double acc = 0.0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) acc += a[i] * b[i];
    const double t = block_sum_256(acc, s_w);
    finalize_sum(t, partials, counter, out);
}

// u -= alpha p ; r -= alpha h ; <r,r>       alpha = rho_res / pdoth   (solve.cpp:2588-2603)
__global__ void __launch_bounds__(256)
pcg_update_kernel(int n, long long ld, double *__restrict__ u, double *__restrict__ r, const double *__restrict__ p,
                  const double *__restrict__ h, const double *__restrict__ scal, int sstride,
                  const int *__restrict__ active, double *partials, unsigned int *counter, double *out_rr) {
    __shared__ double s_w[8];
    const int j = blockIdx.y;
    if (active && !active[j]) return;   // a column that has stopped: every CTA of its row leaves, nothing is reduced
    const long long o = j * ld;
    u += o;
    r += o;
    p += o;
    h += o;
    partials += j * RED_MAX_BLOCKS;
    counter += j;
    out_rr += j;
    const double alpha = scal[S_RHO_RES * sstride + j] / scal[S_PDOTH * sstride + j];
    double acc = 0.0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        u[i] -= alpha * p[i];
        const double ri = r[i] - alpha * h[i];
        r[i] = ri;
        acc += ri * ri;
    }
    const double t = block_sum_256(acc, s_w);
    finalize_sum(t, partials, counter, out_rr);
}

// p = rho + beta p ; beta = <r,rho>_new / rho_res_old ; then rho_res <- <r,rho>_new
// (solve.cpp:2655-2667; the next iteration's <r,rho> at :2580 is the same number, r and rho
// being untouched in between, so it is carried over instead of recomputed)
__global__ void __launch_bounds__(256)
pcg_p_update_kernel(int n, long long ld, double *__restrict__ p, const double *__restrict__ rho,
                    const double *__restrict__ scal, int sstride, const int *__restrict__ active) {
    const int j = blockIdx.y;
    if (active && !active[j]) return;
    p += j * ld;
    rho += j * ld;
    const double beta = scal[S_BETA_NUM * sstride + j] / scal[S_RHO_RES * sstride + j];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        p[i] = rho[i] + beta * p[i];
}

__global__ void carry_scalar_kernel(double *scal, int dst, int src) { scal[dst] = scal[src]; }

// unpreconditioned CG direction update: p = r + (num/den) p
__global__ void __launch_bounds__(256)
cg_p_update_kernel(int n, double *__restrict__ p, const double *__restrict__ r, const double *__restrict__ scal,
                   int num_slot, int den_slot) {
    const double beta = scal[num_slot] / scal[den_slot];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        p[i] = r[i] + beta * p[i];
}

// solve_coarsest_CG's update (saena_object_solve.cpp:58-72): u += f dir; res -= f A dir; <res,res>
__global__ void __launch_bounds__(256)
ccg_update_kernel(int n, double *__restrict__ u, double *__restrict__ res, const double *__restrict__ dir,
                  const double *__restrict__ mv, const double *__restrict__ scal, double *partials,
                  unsigned int *counter, double *out_rr) {
    __shared__ double s_w[8];
    const double factor = scal[S_C_RR] / scal[S_C_DEN];
    double acc = 0.0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        u[i] += factor * dir[i];
        const double ri = res[i] - factor * mv[i];
        res[i] = ri;
        acc += ri * ri;
    }
    const double t = block_sum_256(acc, s_w);
    finalize_sum(t, partials, counter, out_rr);
}

// first Chebyshev sweep from a zero iterate: A*0 = 0, so d = (1/theta) D^-1 rhs and u = d
// (saena_matrix.cpp:1099-1109 with u == 0; bit-identical to running the SpMV on zeros); V = float: the FP32 V-cycle's
template <typename V>
__global__ void __launch_bounds__(256)
cheb_first_zero_kernel(int n, long long ld, const V *__restrict__ rhs, const V *__restrict__ inv_diag,
                       V c, V *__restrict__ d, V *__restrict__ u) {
    const long long o = blockIdx.y * ld;
    rhs += o;
    d += o;
    u += o;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const V v = c * inv_diag[i] * rhs[i];
        d[i] = v;
        u[i] = v;
    }
}

// saena_object::scale_vector (src/saena_object.cpp:563-569)
__global__ void __launch_bounds__(256)
scale_vector_kernel(int n, long long ld, double *__restrict__ v, const double *__restrict__ w) {
    v += blockIdx.y * ld;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) v[i] *= w[i];
}

template <typename V>
__global__ void __launch_bounds__(256)
negate_copy_kernel(int n, long long ld, const V *__restrict__ src, V *__restrict__ dst) {
    src += blockIdx.y * ld;
    dst += blockIdx.y * ld;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) dst[i] = -src[i];
}

// ---------------------------------------------------------------------------------------------
// coarsest level: u = Ainv b, then one refinement step r = b - A u, u += Ainv r.
// One CTA; n is ~100 (least_row_threshold, saena_object.h:43).  Warp per row, rows strided.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
coarsest_kernel(int n, const double *__restrict__ A, const double *__restrict__ Ainv, const double *__restrict__ b,
                double *__restrict__ u, double *__restrict__ tmp) {
    extern __shared__ double s_vec[];  // [n]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    double *x0 = tmp, *r = tmp + n;
    for (int i = threadIdx.x; i < n; i += blockDim.x) s_vec[i] = b[i];
    __syncthreads();
    for (int i = warp; i < n; i += nwarp) {  // x0 = Ainv b
        double s = 0.0;
        for (int j = lane; j < n; j += 32) s += Ainv[(size_t)i * n + j] * s_vec[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) x0[i] = s;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) s_vec[i] = x0[i];
    __syncthreads();
    for (int i = warp; i < n; i += nwarp) {  // r = b - A x0
        double s = 0.0;
        for (int j = lane; j < n; j += 32) s += A[(size_t)i * n + j] * s_vec[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) r[i] = b[i] - s;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) s_vec[i] = r[i];
    __syncthreads();
    for (int i = warp; i < n; i += nwarp) {  // u = x0 + Ainv r
        double s = 0.0;
        for (int j = lane; j < n; j += 32) s += Ainv[(size_t)i * n + j] * s_vec[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) u[i] = x0[i] + s;
    }
}

// ---------------------------------------------------------------------------------------------
// host wrappers
// ---------------------------------------------------------------------------------------------
int sb_dot(saena_b200_ctx *ctx, const double *a, const double *b, int n, int slot) {
    ++ctx->launches;
    dot_kernel<<<red_blocks(ctx, n), 256, 0, ctx->stream>>>(n, 0, a, b, ctx->red_partials, ctx->red_counter,
                                                           ctx->scalars + slot);
    SB_CUDA(cudaGetLastError());
    if (ctx->nranks > 1) SB_TRY(sb_allreduce_sum(ctx, ctx->scalars + slot, 1, ctx->stream));
    return 0;
}

int sb_pcg_update(saena_b200_ctx *ctx, int n, double *u, double *r, const double *p, const double *h) {
    ++ctx->launches;
    pcg_update_kernel<<<red_blocks(ctx, n), 256, 0, ctx->stream>>>(n, 0, u, r, p, h, ctx->scalars, 1, nullptr,
                                                                  ctx->red_partials, ctx->red_counter,
                                                                  ctx->scalars + S_RR);
    SB_CUDA(cudaGetLastError());
    if (ctx->nranks > 1) SB_TRY(sb_allreduce_sum(ctx, ctx->scalars + S_RR, 1, ctx->stream));
    return 0;
}

int sb_pcg_p_update(saena_b200_ctx *ctx, int n, double *p, const double *rho) {
    ctx->launches += 2;
    pcg_p_update_kernel<<<red_blocks(ctx, n), 256, 0, ctx->stream>>>(n, 0, p, rho, ctx->scalars, 1, nullptr);
    carry_scalar_kernel<<<1, 1, 0, ctx->stream>>>(ctx->scalars, S_RHO_RES, S_BETA_NUM);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int sb_cg_p_update(saena_b200_ctx *ctx, int n, double *p, const double *r, int num_slot, int den_slot) {
    ++ctx->launches;
    cg_p_update_kernel<<<red_blocks(ctx, n), 256, 0, ctx->stream>>>(n, p, r, ctx->scalars, num_slot, den_slot);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int sb_cheb_first_zero(saena_b200_ctx *ctx, int n, const double *rhs, const double *inv_diag, double c, double *d,
                       double *u) {
    if (n == 0) return 0;
    ++ctx->launches;
    cheb_first_zero_kernel<<<red_blocks(ctx, n), 256, 0, ctx->stream>>>(n, 0, rhs, inv_diag, c, d, u);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int sb_negate_copy(saena_b200_ctx *ctx, int n, const double *src, double *dst) {
    if (n == 0) return 0;
    ++ctx->launches;
    negate_copy_kernel<<<red_blocks(ctx, n), 256, 0, ctx->stream>>>(n, 0, src, dst);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int sb_cheb_first_zero(saena_b200_ctx *ctx, int n, const float *rhs, const float *inv_diag, float c, float *d, float *u) {
    if (n == 0) return 0;
    ++ctx->launches;
    cheb_first_zero_kernel<<<red_blocks(ctx, n), 256, 0, ctx->stream>>>(n, 0, rhs, inv_diag, c, d, u);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int sb_negate_copy(saena_b200_ctx *ctx, int n, const float *src, float *dst) {
    if (n == 0) return 0;
    ++ctx->launches;
    negate_copy_kernel<<<red_blocks(ctx, n), 256, 0, ctx->stream>>>(n, 0, src, dst);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int sb_fill_zero(saena_b200_ctx *ctx, float *p, size_t n) {
    if (n) SB_CUDA(cudaMemsetAsync(p, 0, n * sizeof(float), ctx->stream));
    return 0;
}

int sb_scale_vector(saena_b200_ctx *ctx, int n, double *v, const double *w) {
    if (n == 0) return 0;
    if (!w) SB_FAIL("scale=true but a level has no inv_sq_diag_orig (saena_b200_upload_level_scale)");
    ++ctx->launches;
    scale_vector_kernel<<<red_blocks(ctx, n), 256, 0, ctx->stream>>>(n, 0, v, w);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int sb_fill_zero(saena_b200_ctx *ctx, double *p, size_t n) {
    if (n) SB_CUDA(cudaMemsetAsync(p, 0, n * sizeof(double), ctx->stream));
    return 0;
}

int sb_coarsest_apply(saena_b200_ctx *ctx, const double *rhs, double *u) {
    const int n = ctx->coarse_n;
    if (n == 0) return 0;
    if (!ctx->coarse_Ainv) SB_FAIL("coarsest solve: no factor uploaded");
    ++ctx->launches;
    const int threads = n >= 512 ? 1024 : (n >= 128 ? 512 : 256);
    coarsest_kernel<<<1, threads, (size_t)n * sizeof(double), ctx->stream>>>(n, ctx->coarse_A, ctx->coarse_Ainv, rhs,
                                                                            u, ctx->coarse_tmp);
    SB_CUDA(cudaGetLastError());
    return 0;
}

// saena_object::solve_coarsest_CG (src/saena_object_solve.cpp:14-114): plain CG on the coarsest
// operator, at most CG_coarsest_max_iter - 1 = 149 iterations, stop at <res,res> < <rhs,rhs> * 1e-24.
// Not the default (direct_solver = "SuperLU", saena_object.h:165); one host read per iteration.
int sb_coarsest_cg(saena_b200_ctx *ctx, const double *rhs, double *u) {
    DevLevel &lv = ctx->levels.back();
    const int n = lv.M;
    if (n == 0) return 0;
    if (ctx->ccg_cap < n) {
        cudaFree(ctx->ccg_res); cudaFree(ctx->ccg_dir); cudaFree(ctx->ccg_mv);
        SB_CUDA(cudaMalloc((void **)&ctx->ccg_res, sizeof(double) * n));
        SB_CUDA(cudaMalloc((void **)&ctx->ccg_dir, sizeof(double) * n));
        SB_CUDA(cudaMalloc((void **)&ctx->ccg_mv, sizeof(double) * n));
        ctx->ccg_cap = n;
    }
    const double tol = 1e-12;  // CG_coarsest_tol, saena_object.h:156
    int max_iter = 150;        // CG_coarsest_max_iter, saena_object.h:155
    double *res = ctx->ccg_res, *dir = ctx->ccg_dir, *mv = ctx->ccg_mv;
    SB_CUDA(cudaMemcpyAsync(res, rhs, sizeof(double) * n, cudaMemcpyDeviceToDevice, ctx->stream));
    SB_CUDA(cudaMemcpyAsync(dir, rhs, sizeof(double) * n, cudaMemcpyDeviceToDevice, ctx->stream));
    SB_TRY(sb_dot(ctx, res, res, n, S_C_RR));
    SB_TRY(sb_read_scalars(ctx));
    const double initial_dot = ctx->scalars_host[S_C_RR];
    const double thres = initial_dot * tol * tol;
    if (initial_dot < tol * tol) max_iter = 0;
    int i = 1;
    while (i < max_iter) {
        EpiArgs e{};
        e.out = mv;
        SB_TRY(sb_apply(ctx, lv.A, dir, EPI_PLAIN, e));
        SB_TRY(sb_dot(ctx, dir, mv, n, S_C_DEN));
        ++ctx->launches;
        ccg_update_kernel<<<red_blocks(ctx, n), 256, 0, ctx->stream>>>(n, u, res, dir, mv, ctx->scalars,
                                                                      ctx->red_partials, ctx->red_counter,
                                                                      ctx->scalars + S_C_RRNEW);
        SB_CUDA(cudaGetLastError());
        SB_TRY(sb_read_scalars(ctx));
        if (ctx->scalars_host[S_C_RRNEW] < thres) break;
        SB_TRY(sb_cg_p_update(ctx, n, dir, res, S_C_RRNEW, S_C_RR));  // dir = res + (dot/dot_prev) dir
        SB_CUDA(cudaMemcpyAsync(ctx->scalars + S_C_RR, ctx->scalars + S_C_RRNEW, sizeof(double),
                                cudaMemcpyDeviceToDevice, ctx->stream));
        i++;
    }
    return 0;
}

// ---- block forms: grid.y = column
static dim3 block_grid(const saena_b200_ctx *ctx, int n, int k) { return dim3(red_blocks(ctx, n), k); }

int sb_dot_block(saena_b200_ctx *ctx, const double *a, const double *b, int n, int k, int slot) {
    ++ctx->launches;
    dot_kernel<<<block_grid(ctx, n, k), 256, 0, ctx->stream>>>(n, n, a, b, ctx->blk_partials, ctx->blk_counter,
                                                              ctx->blk_scal + slot * SB_BLOCK_MAX);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int sb_pcg_update_block(saena_b200_ctx *ctx, int n, int k, double *u, double *r, const double *p, const double *h) {
    ++ctx->launches;
    pcg_update_kernel<<<block_grid(ctx, n, k), 256, 0, ctx->stream>>>(n, n, u, r, p, h, ctx->blk_scal, SB_BLOCK_MAX,
                                                                     ctx->blk_active, ctx->blk_partials,
                                                                     ctx->blk_counter,
                                                                     ctx->blk_scal + S_RR * SB_BLOCK_MAX);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int sb_pcg_p_update_block(saena_b200_ctx *ctx, int n, int k, double *p, const double *rho) {
    ++ctx->launches;
    pcg_p_update_kernel<<<block_grid(ctx, n, k), 256, 0, ctx->stream>>>(n, n, p, rho, ctx->blk_scal, SB_BLOCK_MAX,
                                                                       ctx->blk_active);
    SB_CUDA(cudaGetLastError());
    // rho_res <- <r,rho>_new for every column (a stopped column's are never read again)
    SB_CUDA(cudaMemcpyAsync(ctx->blk_scal + S_RHO_RES * SB_BLOCK_MAX, ctx->blk_scal + S_BETA_NUM * SB_BLOCK_MAX,
                            sizeof(double) * k, cudaMemcpyDeviceToDevice, ctx->stream));
    return 0;
}

int sb_cheb_first_zero_block(saena_b200_ctx *ctx, int n, int k, const double *rhs, const double *inv_diag, double c,
                             double *d, double *u) {
    if (n == 0) return 0;
    ++ctx->launches;
    cheb_first_zero_kernel<<<block_grid(ctx, n, k), 256, 0, ctx->stream>>>(n, n, rhs, inv_diag, c, d, u);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int sb_negate_copy_block(saena_b200_ctx *ctx, int n, int k, const double *src, double *dst) {
    if (n == 0) return 0;
    ++ctx->launches;
    negate_copy_kernel<<<block_grid(ctx, n, k), 256, 0, ctx->stream>>>(n, n, src, dst);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int sb_scale_vector_block(saena_b200_ctx *ctx, int n, int k, double *v, const double *w) {
    if (n == 0) return 0;
    if (!w) SB_FAIL("scale=true but a level has no inv_sq_diag_orig (saena_b200_upload_level_scale)");
    ++ctx->launches;
    scale_vector_kernel<<<block_grid(ctx, n, k), 256, 0, ctx->stream>>>(n, n, v, w);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int sb_read_block_scalars(saena_b200_ctx *ctx) {
    SB_CUDA(cudaMemcpyAsync(ctx->blk_scal_host, ctx->blk_scal, sizeof(double) * S_COUNT * SB_BLOCK_MAX,
                            cudaMemcpyDeviceToHost, ctx->stream));
    return sb_sync_stream(ctx, ctx->stream);
}

int sb_read_scalars(saena_b200_ctx *ctx) {
    // the halo fault words follow the scalars (common.h): the host learns of a timed-out exchange with the same copy
    SB_CUDA(cudaMemcpyAsync(ctx->scalars_host, ctx->scalars, (S_COUNT + S_FAULT_WORDS) * sizeof(double),
                            cudaMemcpyDeviceToHost, ctx->stream));
    return sb_sync_stream(ctx, ctx->stream);
}

// ---------------------------------------------------------------------------------------------
// NVTX ranges (see common.h)
// ---------------------------------------------------------------------------------------------
SbRange::SbRange(const saena_b200_ctx *ctx, const char *name, int level) : on(ctx->nvtx) {
    if (!on) return;
    char buf[64];
    if (level >= 0) snprintf(buf, sizeof(buf), "%s L%d", name, level);
    nvtxRangePushA(level >= 0 ? buf : name);
}
SbRange::~SbRange() {
    if (on) nvtxRangePop();
}
