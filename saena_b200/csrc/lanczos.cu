// lanczos.cu -- the Chebyshev bound of one level on the device: largest eigenvalue of
// D^-1/2 A D^-1/2 by Lanczos, times 1.0001.
//
// SURVEY.md 8f #1 (the component next to the solve path): saena_object::find_eig
// (/root/reference/src/saena_object.cpp:572-590) scales the matrix in place, runs
// find_eig_lamlan (include/lamlan_saena.h:13-79 -> LambdaLanczos::run,
// external/lambda_lanczos/include/lambda_lanczos/lambda_lanczos.hpp:170-260: at most 20 steps,
// full re-orthogonalisation against every earlier Lanczos vector, stop when the Ritz value moves
// by less than 1e-8 relative), stores 1.0001 * lambda in eig_max_of_invdiagXA and scales the matrix
// back.  Here the matrix is not touched: B v = s .* (A (s .* v)), s = sqrt(inv_diag), runs on
// the uploaded operator through the same SpMV kernels (and the same halo exchange on several
// ranks) as the solve; the Ritz value of the small tridiagonal matrix is found on the host by
// bisection on the Sturm count, as the reference does (lambda_lanczos.hpp:303-377).
#include <math.h>

#include <algorithm>
#include <vector>

#include "common.h"

namespace {

__global__ void lz_scaled_copy_kernel(int n, const double *__restrict__ inv_diag, const double *__restrict__ in,
                                      double *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = sqrt(fabs(inv_diag[i])) * in[i];
}

// uk = s .* w - beta * u_prev - alpha * u_cur   (lambda_lanczos.hpp:219-221 with B = S A S)
__global__ void lz_combine_kernel(int n, const double *__restrict__ inv_diag, const double *__restrict__ w, double beta,
                                  const double *__restrict__ u_prev, double alpha, const double *__restrict__ u_cur,
                                  double *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = sqrt(fabs(inv_diag[i])) * w[i] - beta * u_prev[i] - alpha * u_cur[i];
}

// y -= scalars[slot] * x : one Gram-Schmidt step with the inner product still on the device
__global__ void lz_project_out_kernel(int n, const double *__restrict__ scalars, int slot, const double *__restrict__ x,
                                      double *__restrict__ y) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] -= scalars[slot] * x[i];
}

__global__ void lz_scale_kernel(int n, double c, double *__restrict__ y) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] *= c;
}

// start vector: uniform(-1, 1) from a counter-based generator on the GLOBAL row index, so that
// the vector (and the eigenvalue estimate) does not depend on how the rows are partitioned
__global__ void lz_random_kernel(int n, long long row_offset, unsigned long long seed, double *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    unsigned long long z = seed + 0x9E3779B97F4A7C15ull * (unsigned long long)(row_offset + i + 1);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;   // splitmix64
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    out[i] = (double)(z >> 11) * (2.0 / 9007199254740992.0) - 1.0;
}

// number of eigenvalues of the tridiagonal matrix (diagonal a[0..m), off-diagonal b[0..m-1)) below c
int sturm_count(const std::vector<double> &a, const std::vector<double> &b, int m, double c) {
    int count = 0;
    double q = 1.0;
    for (int i = 0; i < m; ++i) {
        const double off = i ? b[i - 1] : 0.0;
        q = a[i] - c - (i ? off * off / q : 0.0);
        if (q < 0.0) ++count;
        if (q == 0.0) q = 1e-15;
    }
    return count;
}

double largest_tridiag_eig(const std::vector<double> &a, const std::vector<double> &b, int m, double rel_eps) {
    double r = 0.0;  // Gershgorin bound
    for (int i = 0; i < m; ++i)
        r = std::max(r, fabs(a[i]) + (i ? fabs(b[i - 1]) : 0.0) + (i + 1 < m ? fabs(b[i]) : 0.0));
    double lo = -r, hi = r, pmid = 1e300;
    while (hi - lo > std::min(fabs(lo), fabs(hi)) * rel_eps) {
        const double mid = 0.5 * (lo + hi);
        if (sturm_count(a, b, m, mid) >= m) hi = mid;  // all m eigenvalues below mid
        else lo = mid;
        if (mid == pmid) break;
        pmid = mid;
    }
    return 0.5 * (lo + hi);
}

}  // namespace

int sb_fill_random(saena_b200_ctx *ctx, int n, long long row_offset, unsigned long long seed, double *out) {
    if (n <= 0) return 0;
    ++ctx->launches;
    lz_random_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(n, row_offset, seed, out);
    SB_CUDA(cudaGetLastError());
    return 0;
}

// eig_out = 1.0001 * lambda_max(D^-1/2 A D^-1/2) of level `level`; start_dev: optional start vector
// (device, this rank's rows), else the seeded generator.  Collective over the ranks.
int sb_find_eig(saena_b200_ctx *ctx, int level, int max_iter, const double *start_dev, unsigned long long seed,
                double *eig_out, int *iters_out) {
    DevLevel &lv = ctx->levels[level];
    const int n = lv.M;
    if (max_iter < 1) max_iter = 20;  // lambda_lanczos.hpp: max_iteration = 20
    const double eps = 1e-8;          // lambda_lanczos.hpp: eps
    const int blocks = std::max(1, (n + 255) / 256);
    cudaStream_t s = ctx->stream;
    // u[0] is the reference's all-zero dummy; u[k] the k-th Lanczos vector; w, t scratch
    std::vector<double *> u;
    double *w = nullptr, *t = nullptr;
    auto release = [&]() {
        for (double *p : u) cudaFree(p);
        cudaFree(w);
        cudaFree(t);
    };
    auto new_vec = [&](double **p) -> int {
        SB_CUDA(cudaMalloc((void **)p, sizeof(double) * std::max(n, 1)));
        return 0;
    };
#define LZ_TRY(expr)            \
    do {                        \
        int rc_ = (expr);       \
        if (rc_) { release(); return rc_; } \
    } while (0)
    LZ_TRY(new_vec(&w));
    LZ_TRY(new_vec(&t));
    for (int k = 0; k < 2; ++k) {
        double *p = nullptr;
        LZ_TRY(new_vec(&p));
        u.push_back(p);
    }
    LZ_TRY(sb_fill_zero(ctx, u[0], n));
    if (start_dev) {
        if (n) cudaMemcpyAsync(u[1], start_dev, sizeof(double) * n, cudaMemcpyDeviceToDevice, s);
    } else {
        LZ_TRY(sb_fill_random(ctx, n, (long long)lv.A.col_offset, seed, u[1]));
    }
    LZ_TRY(sb_dot(ctx, u[1], u[1], n, S_TMP));
    LZ_TRY(sb_read_scalars(ctx));
    if (!(ctx->scalars_host[S_TMP] > 0.0)) { release(); SB_FAIL("find_eig: zero start vector"); }
    if (n) lz_scale_kernel<<<blocks, 256, 0, s>>>(n, 1.0 / sqrt(ctx->scalars_host[S_TMP]), u[1]);

    std::vector<double> alpha, beta;  // alpha[k-1], beta[k-1] of step k
    double betak = 0.0, ev = 0.0, pev = 1e300;
    int itern = max_iter;
    for (int k = 1; k <= max_iter; ++k) {
        // w = A (s .* u_k)
        if (n) lz_scaled_copy_kernel<<<blocks, 256, 0, s>>>(n, lv.inv_diag, u[k], t);
        EpiArgs e{};
        e.out = w;
        LZ_TRY(sb_apply(ctx, lv.A, t, EPI_PLAIN, e));
        // alpha_k = <u_k, s .* w>
        if (n) lz_scaled_copy_kernel<<<blocks, 256, 0, s>>>(n, lv.inv_diag, w, t);
        LZ_TRY(sb_dot(ctx, u[k], t, n, S_TMP));
        LZ_TRY(sb_read_scalars(ctx));
        const double alphak = ctx->scalars_host[S_TMP];
        alpha.push_back(alphak);
        // u_{k+1} = B u_k - beta_{k-1} u_{k-1} - alpha_k u_k, then modified Gram-Schmidt against all u
        double *next = nullptr;
        LZ_TRY(new_vec(&next));
        u.push_back(next);
        if (n) lz_combine_kernel<<<blocks, 256, 0, s>>>(n, lv.inv_diag, w, betak, u[k - 1], alphak, u[k], next);
        for (int j = 0; j <= k; ++j) {  // lambda_lanczos_util.hpp:190-200 (u[0] = 0 contributes nothing)
            LZ_TRY(sb_dot(ctx, u[j], next, n, S_TMP));
            if (n) lz_project_out_kernel<<<blocks, 256, 0, s>>>(n, ctx->scalars, S_TMP, u[j], next);
        }
        LZ_TRY(sb_dot(ctx, next, next, n, S_TMP));
        LZ_TRY(sb_read_scalars(ctx));
        betak = sqrt(ctx->scalars_host[S_TMP]);
        beta.push_back(betak);
        ev = largest_tridiag_eig(alpha, beta, k, eps * 0.1);  // tridiag_eps_ratio = 1e-1
        if (betak < 1e-16) { itern = k; break; }              // invariant subspace found
        if (n) lz_scale_kernel<<<blocks, 256, 0, s>>>(n, 1.0 / betak, next);
        if (fabs(ev - pev) < std::min(fabs(ev), fabs(pev)) * eps) { itern = k; break; }
        pev = ev;
    }
#undef LZ_TRY
    const int sync_rc = sb_sync_stream(ctx, s);
    release();
    if (sync_rc) return sync_rc;
    SB_TRY(sb_check_fault(ctx));
    *eig_out = 1.0001 * ev;  // lamlan_saena.h:59
    if (iters_out) *iters_out = itern;
    ctx->launches += 4 * itern;
    return 0;
}
