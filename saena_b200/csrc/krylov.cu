// krylov.cu -- the Arnoldi process of the flexible GMRES solve (saena_b200_solve_gmres, api.cu): one step's
// orthogonalisation of w = A z_j against the basis v_0 .. v_j by classical Gram-Schmidt applied twice (CGS2), the
// normalisation of v_{j+1} and the end-of-cycle update x -= Z y.
//
// The basis is one allocation of vectors at a fixed stride ld (a multiple of 32 doubles, so that every vector starts
// 256-byte aligned).  Every kernel is one pass over the vectors it touches, bandwidth-bound:
//   gm_multidot     h1_i = <v_i, w> (i < nv) and <w, w>            reads v_0..v_{nv-1} and w once
//   gm_update_dot   w' = w - V h1, then h2_i = <v_i, w'>, <w', w'>   reads V and w once, writes w (V held in registers)
//   gm_correct      w'' = w' - V h2, <w'', w''>; the last CTA writes the Hessenberg column h1 + h2, ||w''||, ||w||
//   gm_normalize    v_{j+1} = w'' / h and a copy into the preconditioner's input vector
//   gm_multi_axpy   x -= sum_i y_i z_i
// Reductions are deterministic: each thread keeps its running sums in shared memory (one column per thread), a CTA
// sums them in a fixed tree, every CTA writes one partial per sum, and the last CTA to finish (atomic ticket) adds the
// partials in index order -- no floating-point atomics, the grid depends only on n, the number of vectors and the SM
// count, so a repeated call gives the same bits.  The partials, the counter and the scalars are the solve's own
// (ctx->gm_*), shared with no other path.
#include <math.h>

#include <algorithm>

#include "common.h"

static const int GM_THREADS = 128;
static const int GM_SLOTS = SB_GMRES_MAX + 2;   // sums of one reduction: up to 64 dots and one squared norm

// scalar slots of ctx->gm_scal: the three reductions' outputs and the Hessenberg column the host reads
static const int GM_S1 = 0;                   // h1[0..nv), |w|^2 at [nv]
static const int GM_S2 = GM_SLOTS;            // h2[0..nv), |w'|^2 at [nv]
static const int GM_S3 = 2 * GM_SLOTS;        // |w''|^2
static const int GM_COL = 3 * GM_SLOTS;       // column: h1 + h2 [0..nv), |w''| at [nv], |w| at [nv + 1]
static const int GM_SCAL = 4 * GM_SLOTS;

// Reduction of the per-thread sums s_acc[i * blockDim + t] (i < nacc) over the grid into out[i].  One warp per sum,
// lanes over a fixed stride, a fixed shuffle tree: the same order in every call.
__device__ __forceinline__ bool gm_reduce(const double *s_acc, int nacc, double *partials, unsigned int *counter,
                                          double *out) {
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    __syncthreads();
    for (int i = warp; i < nacc; i += nw) {
        double t = 0.0;
        for (int k = lane; k < (int)blockDim.x; k += 32) t += s_acc[i * blockDim.x + k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        if (lane == 0) partials[(size_t)i * RED_MAX_BLOCKS + blockIdx.x] = t;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(counter, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!s_last) return false;
    __threadfence();
    for (int i = warp; i < nacc; i += nw) {
        double t = 0.0;
        for (unsigned int b = lane; b < gridDim.x; b += 32) t += __ldcg(partials + (size_t)i * RED_MAX_BLOCKS + b);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        if (lane == 0) out[i] = t;
    }
    if (threadIdx.x == 0) *counter = 0u;
    __syncthreads();
    return true;   // the last CTA: out[] is complete and visible to its threads
}

__device__ __forceinline__ void gm_zero_acc(double *s_acc, int nacc) {
    for (int i = threadIdx.x; i < nacc * (int)blockDim.x; i += blockDim.x) s_acc[i] = 0.0;
    __syncthreads();
}

// h1_i = <v_i, w> for i < nv, and <w, w> as sum nv
__global__ void __launch_bounds__(GM_THREADS)
gm_multidot_kernel(int n, long long ld, const double *__restrict__ V, int nv, const double *__restrict__ w,
                   double *partials, unsigned int *counter, double *out) {
    extern __shared__ double s_acc[];
    gm_zero_acc(s_acc, nv + 1);
    double *mine = s_acc + threadIdx.x;
    for (int e = blockIdx.x * GM_THREADS + threadIdx.x; e < n; e += gridDim.x * GM_THREADS) {
        const double we = w[e];
#pragma unroll 8
        for (int i = 0; i < nv; ++i) mine[i * GM_THREADS] += V[i * ld + e] * we;
        mine[nv * GM_THREADS] += we * we;
    }
    gm_reduce(s_acc, nv + 1, partials, counter, out);
}

// w' = w - sum_i h_i v_i (in index order), written over w; then h2_i = <v_i, w'> and <w', w'>.  The nv <= J basis
// elements of a row are loaded once into registers and feed both steps.
template <int J>
__global__ void __launch_bounds__(GM_THREADS)
gm_update_dot_kernel(int n, long long ld, const double *__restrict__ V, int nv, double *__restrict__ w,
                     const double *__restrict__ h, double *partials, unsigned int *counter, double *out) {
    extern __shared__ double s_acc[];
    __shared__ double s_h[J];
    for (int i = threadIdx.x; i < J; i += blockDim.x) s_h[i] = i < nv ? h[i] : 0.0;
    gm_zero_acc(s_acc, nv + 1);
    double *mine = s_acc + threadIdx.x;
    // read from shared memory at every use: hoisted out of the row loop, J coefficients would take 2 J registers next
    // to the J basis elements and spill at J = 64
    const volatile double *coef = s_h;
    for (int e = blockIdx.x * GM_THREADS + threadIdx.x; e < n; e += gridDim.x * GM_THREADS) {
        double v[J];
#pragma unroll
        for (int i = 0; i < J; ++i) v[i] = i < nv ? V[i * ld + e] : 0.0;
        double s = w[e];
#pragma unroll
        for (int i = 0; i < J; ++i)
            if (i < nv) s -= coef[i] * v[i];
        w[e] = s;
#pragma unroll
        for (int i = 0; i < J; ++i)
            if (i < nv) mine[i * GM_THREADS] += v[i] * s;
        mine[nv * GM_THREADS] += s * s;
    }
    gm_reduce(s_acc, nv + 1, partials, counter, out);
}

// w'' = w' - sum_i h2_i v_i and <w'', w''>.  The last CTA then writes the Hessenberg column: h1_i + h2_i (i < nv),
// ||w''|| and ||w|| (the norm before the orthogonalisation, from gm_multidot's last sum).
__global__ void __launch_bounds__(GM_THREADS)
gm_correct_kernel(int n, long long ld, const double *__restrict__ V, int nv, double *__restrict__ w,
                  double *scal, double *partials, unsigned int *counter) {
    extern __shared__ double s_acc[];
    __shared__ double s_h[SB_GMRES_MAX];
    const double *h1 = scal + GM_S1, *h2 = scal + GM_S2;
    for (int i = threadIdx.x; i < nv; i += blockDim.x) s_h[i] = h2[i];
    gm_zero_acc(s_acc, 1);
    double acc = 0.0;
    for (int e = blockIdx.x * GM_THREADS + threadIdx.x; e < n; e += gridDim.x * GM_THREADS) {
        double s = w[e];
#pragma unroll 8
        for (int i = 0; i < nv; ++i) s -= s_h[i] * V[i * ld + e];
        w[e] = s;
        acc += s * s;
    }
    s_acc[threadIdx.x] = acc;
    if (!gm_reduce(s_acc, 1, partials, counter, scal + GM_S3)) return;
    double *col = scal + GM_COL;
    for (int i = threadIdx.x; i < nv; i += blockDim.x) col[i] = h1[i] + h2[i];
    if (threadIdx.x == 0) {
        col[nv] = sqrt(scal[GM_S3]);
        col[nv + 1] = sqrt(h1[nv]);
    }
}

// v = v / h in place; t = v (the vector the preconditioner reads)
__global__ void __launch_bounds__(256)
gm_normalize_kernel(int n, double *__restrict__ v, double h, double *__restrict__ t) {
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
        const double x = v[e] / h;
        v[e] = x;
        t[e] = x;
    }
}

struct GmCoef {
    double y[SB_GMRES_MAX];
};

// x -= sum_i y_i z_i, in index order
__global__ void __launch_bounds__(256)
gm_multi_axpy_kernel(int n, long long ld, const double *__restrict__ Z, int k, GmCoef c, double *__restrict__ x) {
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
        double s = x[e];
#pragma unroll 8
        for (int i = 0; i < k; ++i) s -= c.y[i] * Z[i * ld + e];
        x[e] = s;
    }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static size_t acc_bytes(int nacc) { return sizeof(double) * (size_t)nacc * GM_THREADS; }

// CTAs of a reduction pass: as many as fit on the SMs at once at this shared-memory footprint and at most max_per_sm
// (the register limit) per SM, fewer for a short vector.  A function of (n, nacc, SM count) only, so that repeated
// calls reduce in the same order.
static int gm_grid(const saena_b200_ctx *ctx, int n, int nacc, int max_per_sm = 8) {
    int per_sm = (int)((200u << 10) / acc_bytes(nacc));
    per_sm = per_sm < 1 ? 1 : (per_sm > max_per_sm ? max_per_sm : per_sm);
    int b = (n + GM_THREADS - 1) / GM_THREADS;
    const int cap = std::min(ctx->sm_count * per_sm, RED_MAX_BLOCKS);
    return b > cap ? cap : (b < 1 ? 1 : b);
}

static int stream_grid(const saena_b200_ctx *ctx, int n) {
    const int b = (n + 1023) / 1024;
    return std::max(1, std::min(b, ctx->sm_count * 8));
}

void sb_gmres_state_free(saena_b200_ctx *ctx) {
    cudaFree(ctx->gm_partials); ctx->gm_partials = nullptr;
    cudaFree(ctx->gm_counter); ctx->gm_counter = nullptr;
    cudaFree(ctx->gm_scal); ctx->gm_scal = nullptr;
    cudaFreeHost(ctx->gm_scal_host); ctx->gm_scal_host = nullptr;
}

int sb_gmres_state(saena_b200_ctx *ctx) {
    if (ctx->gm_scal_host) return 0;
    bool ok = cudaMalloc((void **)&ctx->gm_partials, sizeof(double) * GM_SLOTS * RED_MAX_BLOCKS) == cudaSuccess &&
              cudaMalloc((void **)&ctx->gm_counter, sizeof(unsigned int)) == cudaSuccess &&
              cudaMemsetAsync(ctx->gm_counter, 0, sizeof(unsigned int), ctx->stream) == cudaSuccess &&
              cudaMalloc((void **)&ctx->gm_scal, sizeof(double) * GM_SCAL) == cudaSuccess &&
              cudaMemsetAsync(ctx->gm_scal, 0, sizeof(double) * GM_SCAL, ctx->stream) == cudaSuccess &&
              cudaMallocHost((void **)&ctx->gm_scal_host, sizeof(double) * GM_SCAL) == cudaSuccess;
    // the reductions of the widest steps need more than the default 48 KB of shared memory per CTA
    const int big = (int)acc_bytes(GM_SLOTS);
    ok = ok && cudaFuncSetAttribute(gm_multidot_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, big) == cudaSuccess &&
         cudaFuncSetAttribute(gm_update_dot_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, big) == cudaSuccess &&
         cudaFuncSetAttribute(gm_update_dot_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, big) == cudaSuccess &&
         cudaFuncSetAttribute(gm_update_dot_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, big) == cudaSuccess &&
         cudaFuncSetAttribute(gm_update_dot_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, big) == cudaSuccess;
    if (!ok) {
        cudaGetLastError();   // an out-of-memory status is not sticky
        sb_gmres_state_free(ctx);
        SB_FAIL("gmres: not enough device memory for the reduction state");
    }
    return 0;
}

int sb_gmres_norm2(saena_b200_ctx *ctx, int n, const double *w) {
    ++ctx->launches;
    gm_multidot_kernel<<<gm_grid(ctx, n, 1), GM_THREADS, acc_bytes(1), ctx->stream>>>(
        n, 0, nullptr, 0, w, ctx->gm_partials, ctx->gm_counter, ctx->gm_scal + GM_S1);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int sb_gmres_orthogonalize(saena_b200_ctx *ctx, int n, long long ld, const double *V, int nv, double *w) {
    if (nv < 0 || nv > SB_GMRES_MAX) SB_FAIL("gmres: basis size out of range");
    const int nacc = nv + 1;
    const size_t sm = acc_bytes(nacc);
    const int grid = gm_grid(ctx, n, nacc);
    // gm_update_dot's registers (sm_100a, -Xptxas -v): 39 / 64 / 104 / 177 for J = 8 / 16 / 32 / 64, so 8 / 8 / 4 / 2
    // CTAs of 128 threads per SM
    const int grid_upd = gm_grid(ctx, n, nacc, nv <= 16 ? 8 : (nv <= 32 ? 4 : 2));
    double *part = ctx->gm_partials, *scal = ctx->gm_scal;
    unsigned int *cnt = ctx->gm_counter;
    ctx->launches += 3;
    gm_multidot_kernel<<<grid, GM_THREADS, sm, ctx->stream>>>(n, ld, V, nv, w, part, cnt, scal + GM_S1);
    if (nv <= 8)
        gm_update_dot_kernel<8><<<grid_upd, GM_THREADS, sm, ctx->stream>>>(n, ld, V, nv, w, scal + GM_S1, part, cnt, scal + GM_S2);
    else if (nv <= 16)
        gm_update_dot_kernel<16><<<grid_upd, GM_THREADS, sm, ctx->stream>>>(n, ld, V, nv, w, scal + GM_S1, part, cnt, scal + GM_S2);
    else if (nv <= 32)
        gm_update_dot_kernel<32><<<grid_upd, GM_THREADS, sm, ctx->stream>>>(n, ld, V, nv, w, scal + GM_S1, part, cnt, scal + GM_S2);
    else
        gm_update_dot_kernel<64><<<grid_upd, GM_THREADS, sm, ctx->stream>>>(n, ld, V, nv, w, scal + GM_S1, part, cnt, scal + GM_S2);
    gm_correct_kernel<<<gm_grid(ctx, n, 1), GM_THREADS, acc_bytes(1), ctx->stream>>>(n, ld, V, nv, w, scal, part, cnt);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int sb_gmres_normalize(saena_b200_ctx *ctx, int n, double *v, double h, double *t) {
    if (n == 0) return 0;
    ++ctx->launches;
    gm_normalize_kernel<<<stream_grid(ctx, n), 256, 0, ctx->stream>>>(n, v, h, t);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int sb_gmres_update(saena_b200_ctx *ctx, int n, long long ld, const double *Z, int k, const double *y, double *x) {
    if (n == 0 || k == 0) return 0;
    if (k > SB_GMRES_MAX) SB_FAIL("gmres: update of more than 64 vectors");
    GmCoef c{};
    for (int i = 0; i < k; ++i) c.y[i] = y[i];
    ++ctx->launches;
    gm_multi_axpy_kernel<<<stream_grid(ctx, n), 256, 0, ctx->stream>>>(n, ld, Z, k, c, x);
    SB_CUDA(cudaGetLastError());
    return 0;
}

// gm_scal -> gm_scal_host (synchronises the stream)
int sb_gmres_read(saena_b200_ctx *ctx) {
    SB_CUDA(cudaMemcpyAsync(ctx->gm_scal_host, ctx->gm_scal, sizeof(double) * GM_SCAL, cudaMemcpyDeviceToHost,
                            ctx->stream));
    return sb_sync_stream(ctx, ctx->stream);
}

double sb_gmres_norm2_host(const saena_b200_ctx *ctx) { return ctx->gm_scal_host[GM_S1]; }
const double *sb_gmres_h1_host(const saena_b200_ctx *ctx) { return ctx->gm_scal_host + GM_S1; }
const double *sb_gmres_h2_host(const saena_b200_ctx *ctx) { return ctx->gm_scal_host + GM_S2; }
const double *sb_gmres_column_host(const saena_b200_ctx *ctx) { return ctx->gm_scal_host + GM_COL; }
