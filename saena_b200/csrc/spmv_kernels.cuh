// spmv_kernels.cuh -- FP64 / int32-column CSR SpMV kernels for sm_100a with fused epilogues.
//
// Replaces the scalar loops of saena_matrix::matvec_sparse (/root/reference/src/
// saena_matrix_matvec.cpp:68-80 local part, :87-110 remote part), the residual variants of
// include/saena_matrix.tpp:16-43 and the update loops of saena_matrix::chebyshev / jacobi
// (src/saena_matrix.cpp:1044-1131).  All of it is HBM-bound (<= 0.17 flop/byte): no tensor
// cores; what matters is that every byte of val/col/vectors is fetched once, in full 128-byte
// lines, with enough loads in flight.
//
// Three row mappings, chosen per operator from nnz/row and row-length regularity (sb_choose_mapping):
//   spmv_sell          32-row slices stored column-major (padded per slice): lane = row, every load
//                      coalesced and independent.  Short regular rows (the 7-point level 0).
//   spmv_symdiag<ND>   an exactly symmetric operator on a few diagonals: diagonal 0 and the positive
//                      offsets as dense arrays, no column ids.  The 7-point level 0 on one rank.
//   spmv_rowgroup<TPR> 32..256 threads per row: the deep coarse levels (thousands of nnz per row)
//   spmv_vec<LANES>    LANES (1..16) lanes cooperate on a row, a warp owns 32 consecutive rows
//                      and results are transposed so lane j finishes row j: the epilogue's
//                      vector streams (rhs, inv_diag, d, u) are read and written fully coalesced.
//   spmv_stream<LPR>   a CTA owns a block of consecutive rows holding <= STREAM_TILE non-zeros;
//                      val/col are streamed in perfectly coalesced order, products go to shared
//                      memory, then LPR lanes per row reduce their segment.  Best for short rows
//                      (7-point level 0) where a per-row mapping wastes lanes.
#pragma once

#include <type_traits>

#include "common.h"

// Every input of row i is read before the first store: the pointers are not restrict-qualified, so a load written after
// a store is issued only once the values the store depends on have arrived -- a second memory round trip per thread.
// (No caller passes u_in aliasing d_out; out may be u_in, d_out may be d_in: same element, read first either way.)
// Row i of the operator; o: where row i's entries of the epilogue's vectors are (i, or i + j * ld in column j of a
// block: inv_diag, one per row, is shared by the columns).
// V: the value type (double; float in the FP32 preconditioner's instantiations, spmv_f32.cu).
template <int EPI, typename IdxT, typename V>
__device__ __forceinline__ void sb_epilogue_at(int i, IdxT o, V ax, const EpiArgsT<V> &e) {
    if (EPI == EPI_PLAIN) {
        e.out[o] = ax;
    } else if (EPI == EPI_RESIDUAL) {
        e.out[o] = ax - e.rhs[o];
    } else if (EPI == EPI_CHEB_FIRST) {
        const V u = e.u_in[o];
        const V d = e.c1 * e.inv_diag[i] * (e.rhs[o] - ax);
        e.d_out[o] = d;
        e.out[o] = u + d;
    } else if (EPI == EPI_CHEB_NEXT) {
        const V u = e.u_in[o];
        const V res = e.c2 * e.inv_diag[i] * (e.rhs[o] - ax);
        const V d = (e.c1 * e.d_in[o]) + res;
        e.d_out[o] = d;
        e.out[o] = u + d;
    } else if (EPI == EPI_JACOBI) {
        const V t = (ax - e.rhs[o]) * (e.inv_diag[i] * e.c1);
        e.out[o] = e.u_in[o] - t;
    } else if (EPI == EPI_SUB) {
        e.out[o] = e.u_in[o] - ax;
    }
}

template <int EPI, typename V>
__device__ __forceinline__ void sb_epilogue(int i, V ax, const EpiArgsT<V> &e) {
    sb_epilogue_at<EPI>(i, i, ax, e);
}

// (Fetching the epilogue's vector inputs before the row loop was tried in round 1: +3 % on the
// 7-point level, -12 %/-20 % on the 68 and 267 nnz/row levels -- the extra live registers cost the
// loop its load batching at 32 registers/thread.  Not adopted.)
__device__ __forceinline__ bool sb_row_skipped(const uint32_t *__restrict__ mask, int row) {
    return mask != nullptr && ((mask[row >> 5] >> (row & 31)) & 1u);
}

// streaming loads of the matrix arrays: read once, do not pollute L1
__device__ __forceinline__ double sb_ld_stream(const double *p) { return __ldcs(p); }
__device__ __forceinline__ int sb_ld_stream(const int *p) { return __ldcs(p); }
__device__ __forceinline__ float sb_ld_stream(const float *p) { return __ldcs(p); }

// Where the gathered operand comes from.  XLocal: the rank's own vector.  XGhost (merged mode of the
// fused halo kernel, csrc/fused_halo.cu): columns >= n_local are ghost values the neighbours stored
// into this rank's landing area over NVLink.  Plain (L1-cached) loads: the gather reuses ghost
// values across rows as much as local ones (deep levels: thousands of entries per row), and no
// line of the landing area can be stale in L1 -- L1 is invalidated at every launch and within a
// launch nothing reads the area before the `arrived` flag has been observed.
template <typename V>
struct XLocalT {
    const V *x;
    __device__ __forceinline__ V ld(int c) const { return __ldg(x + c); }
};
using XLocal = XLocalT<double>;
struct XGhost {
    const double *x;
    const double *ghost;
    int n_local;
    __device__ __forceinline__ double ld(int c) const {
        const double *p = c < n_local ? x + c : ghost + (c - n_local);  // one load from a selected address: no branch
        return *p;
    }
};

// Every mapping is a __device__ body taking the CTA's index as an argument (`vb`), wrapped by a
// plain __global__ kernel (one operator application on one rank) and reused by the fused halo
// kernel, where a CTA's role -- pack, interior rows, rows waiting for ghost values -- depends on
// its index.
// ---------------------------------------------------------------------------------------------
// spmv_vec: LANES lanes per row, warp = 32 consecutive rows, transposed epilogue
// ---------------------------------------------------------------------------------------------
constexpr int VEC_UNROLL = 4;

template <int LANES, int EPI, typename OffT, typename XS, typename V>
__device__ __forceinline__ void
spmv_vec_body(int vb, int row_begin, int M, const OffT *__restrict__ rowptr, const int *__restrict__ col,
              const V *__restrict__ val, const XS xs, const EpiArgsT<V> &e,
              const uint32_t *__restrict__ skip_mask) {
    constexpr int G = 32 / LANES;  // rows in flight per warp per step
    const int lane = threadIdx.x & 31;
    const int warp = (vb * blockDim.x + threadIdx.x) >> 5;
    const int row0 = row_begin + warp * 32;  // rows [row_begin, M)
    if (row0 >= M) return;
    const int my_row = row0 + lane;
    // lane j fetches the extent of row j (coalesced), shuffled to the cooperating lanes below
    OffT my_start = 0, my_end = 0;
    if (my_row < M) {
        my_start = rowptr[my_row];
        my_end = rowptr[my_row + 1];
    }
    V mine = V(0);
    const int g = lane / LANES;   // which row of the step this lane works on
    const int sub = lane % LANES;
#pragma unroll
    for (int t = 0; t < LANES; ++t) {
        const int src = t * G + g;  // lane that owns the row this group works on in step t
        const OffT start = __shfl_sync(0xffffffffu, my_start, src);
        const OffT end = __shfl_sync(0xffffffffu, my_end, src);
        V sum = V(0);
        for (OffT k = start + sub; k < end; k += LANES * VEC_UNROLL) {
            // issue all loads of the trip before the first use: VEC_UNROLL independent chains
            int c[VEC_UNROLL];
            V a[VEC_UNROLL];
#pragma unroll
            for (int q = 0; q < VEC_UNROLL; ++q) {
                const OffT kk = k + q * LANES;
                const bool in = kk < end;
                c[q] = in ? sb_ld_stream(col + kk) : 0;
                a[q] = in ? sb_ld_stream(val + kk) : V(0);
            }
#pragma unroll
            for (int q = 0; q < VEC_UNROLL; ++q) sum += a[q] * xs.ld(c[q]);
        }
#pragma unroll
        for (int o = LANES / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        // lane j = t*G + g' wants the sum of group g' = j % G
        const V v = __shfl_sync(0xffffffffu, sum, (lane % G) * LANES);
        if (lane / G == t) mine = v;
    }
    if (my_row < M && !sb_row_skipped(skip_mask, my_row)) sb_epilogue<EPI>(my_row, mine, e);
}

template <int LANES, int EPI, typename OffT, typename V = double>
__global__ void __launch_bounds__(256)
spmv_vec_kernel(int row_begin, int M, const OffT *__restrict__ rowptr, const int *__restrict__ col,
                const V *__restrict__ val, const V *__restrict__ x, EpiArgsT<V> e,
                const uint32_t *__restrict__ skip_mask) {
    spmv_vec_body<LANES, EPI, OffT>(blockIdx.x, row_begin, M, rowptr, col, val, XLocalT<V>{x}, e, skip_mask);
}

// ---------------------------------------------------------------------------------------------
// spmv_rowgroup: TPR = 32..256 threads per row, 256/TPR rows per CTA.  For the deep coarse levels
// of a smoothed-aggregation hierarchy: a few thousand rows with thousands of non-zeros each
// (256^3 Poisson: level 4 has 21 466 rows x 3025 nnz/row).  One row per warp-group keeps all SMs
// busy where the 32-rows-per-warp mapping above would leave most of the chip idle.
// ---------------------------------------------------------------------------------------------
template <int TPR, int EPI, typename OffT, typename XS, typename V>
__device__ __forceinline__ void
spmv_rowgroup_body(int vb, int row_begin, int M, const OffT *__restrict__ rowptr, const int *__restrict__ col,
                   const V *__restrict__ val, const XS xs, const EpiArgsT<V> &e,
                   const uint32_t *__restrict__ skip_mask) {
    constexpr int ROWS = 256 / TPR;
    constexpr int WPR = TPR / 32;  // warps per row
    __shared__ V s_part[8];
    const int g = threadIdx.x / TPR, sub = threadIdx.x % TPR;
    const int row = row_begin + vb * ROWS + g;  // rows [row_begin, M)
    V sum = V(0);
    if (row < M) {
        const OffT start = rowptr[row], end = rowptr[row + 1];
        for (OffT k = start + sub; k < end; k += TPR * VEC_UNROLL) {
            int c[VEC_UNROLL];
            V a[VEC_UNROLL];
#pragma unroll
            for (int q = 0; q < VEC_UNROLL; ++q) {
                const OffT kk = k + q * TPR;
                const bool in = kk < end;
                c[q] = in ? sb_ld_stream(col + kk) : 0;
                a[q] = in ? sb_ld_stream(val + kk) : V(0);
            }
#pragma unroll
            for (int q = 0; q < VEC_UNROLL; ++q) sum += a[q] * xs.ld(c[q]);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (WPR == 1) {
        if (sub == 0 && row < M && !sb_row_skipped(skip_mask, row)) sb_epilogue<EPI>(row, sum, e);
    } else {
        if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = sum;
        __syncthreads();
        if (sub == 0 && row < M && !sb_row_skipped(skip_mask, row)) {
            V tot = V(0);
#pragma unroll
            for (int w = 0; w < WPR; ++w) tot += s_part[g * WPR + w];
            sb_epilogue<EPI>(row, tot, e);
        }
    }
}

template <int TPR, int EPI, typename OffT, typename V = double>
__global__ void __launch_bounds__(256)
spmv_rowgroup_kernel(int row_begin, int M, const OffT *__restrict__ rowptr, const int *__restrict__ col,
                     const V *__restrict__ val, const V *__restrict__ x, EpiArgsT<V> e,
                     const uint32_t *__restrict__ skip_mask) {
    spmv_rowgroup_body<TPR, EPI, OffT>(blockIdx.x, row_begin, M, rowptr, col, val, XLocalT<V>{x}, e, skip_mask);
}

// ---------------------------------------------------------------------------------------------
// spmv_stream: CTA = block of consecutive rows with <= STREAM_TILE nnz
// ---------------------------------------------------------------------------------------------
template <int LPR, int EPI, typename OffT>
__global__ void __launch_bounds__(STREAM_THREADS)
spmv_stream_kernel(int M, const OffT *__restrict__ rowptr, const int *__restrict__ col,
                   const double *__restrict__ val, const double *__restrict__ x, EpiArgs e,
                   const uint32_t *__restrict__ skip_mask, const int *__restrict__ blk_row) {
    constexpr int ROWS = STREAM_THREADS / LPR;  // max rows per block
    __shared__ double s_prod[STREAM_TILE];
    __shared__ OffT s_rp[STREAM_THREADS + 1];
    __shared__ double s_red[STREAM_THREADS / 32];
    const int tid = threadIdx.x;
    const int r0 = blk_row[blockIdx.x];
    const int r1 = blk_row[blockIdx.x + 1];
    const int nrows = r1 - r0;  // <= ROWS
    for (int i = tid; i <= nrows; i += STREAM_THREADS) s_rp[i] = rowptr[r0 + i];
    __syncthreads();
    const OffT base = s_rp[0];
    const OffT nnzb = s_rp[nrows] - base;

    if (nnzb > STREAM_TILE) {
        // a single row longer than the tile (the host puts such a row alone in its block)
        double sum = 0.0;
        for (OffT k = tid; k < nnzb; k += STREAM_THREADS)
            sum += sb_ld_stream(val + base + k) * __ldg(x + sb_ld_stream(col + base + k));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        if ((tid & 31) == 0) s_red[tid >> 5] = sum;
        __syncthreads();
        if (tid == 0) {
            double tot = 0.0;
            for (int w = 0; w < STREAM_THREADS / 32; ++w) tot += s_red[w];
            if (!sb_row_skipped(skip_mask, r0)) sb_epilogue<EPI>(r0, tot, e);
        }
        return;
    }

    // phase 1: products in storage order -- every load is a full coalesced line
    const int n = (int)nnzb;
    {
        constexpr int U = STREAM_TILE / STREAM_THREADS;  // every thread's share of a full tile
        int c[U];
        double a[U];
#pragma unroll
        for (int q = 0; q < U; ++q) {  // all loads of the tile in flight before the first use
            const int k = tid + q * STREAM_THREADS;
            const bool in = k < n;
            c[q] = in ? sb_ld_stream(col + base + k) : 0;
            a[q] = in ? sb_ld_stream(val + base + k) : 0.0;
        }
#pragma unroll
        for (int q = 0; q < U; ++q) {
            const int k = tid + q * STREAM_THREADS;
            if (k < n) s_prod[k] = a[q] * __ldg(x + c[q]);
        }
    }
    __syncthreads();

    // phase 2: LPR lanes reduce one row's segment
    if (LPR == 1) {
        if (tid < nrows) {
            const int a = (int)(s_rp[tid] - base), b = (int)(s_rp[tid + 1] - base);
            double sum = 0.0;
            for (int k = a; k < b; ++k) sum += s_prod[k];
            const int row = r0 + tid;
            if (!sb_row_skipped(skip_mask, row)) sb_epilogue<EPI>(row, sum, e);
        }
    } else {
        __shared__ double s_rowsum[ROWS];
        const int rr = tid / LPR, sub = tid % LPR;
        double sum = 0.0;
        if (rr < nrows) {
            const int a = (int)(s_rp[rr] - base), b = (int)(s_rp[rr + 1] - base);
            for (int k = a + sub; k < b; k += LPR) sum += s_prod[k];
        }
#pragma unroll
        for (int o = LPR / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        if (sub == 0 && rr < nrows) s_rowsum[rr] = sum;
        __syncthreads();
        if (tid < nrows) {
            const int row = r0 + tid;
            if (!sb_row_skipped(skip_mask, row)) sb_epilogue<EPI>(row, s_rowsum[tid], e);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// spmv_sell: sliced layout for short, regular rows (the 7-point level 0).  At upload the CSR
// rows are regrouped in slices of 32 consecutive rows, each slice stored column-major and padded
// to its longest row (val 0.0, col = the row's own last column), still FP64 values / int32
// columns.  Lane t owns row t of the slice: the j-th entries of the 32 rows are one 256-byte and
// one 128-byte line, every load of the loop is independent and fully coalesced, and for a
// stencil the x gather is coalesced too (neighbour j of 32 consecutive rows = 32 consecutive x).
// No shuffles, no shared memory; the epilogue streams are coalesced by construction.
// ---------------------------------------------------------------------------------------------
// One lane's row of a slice of `len` entries (cp, vp: the lane's first entry), summed in column order.  Each trip
// covers DEPTH entries, its loads predicated on the slice's length -- the same for all 32 lanes, so nothing diverges.
// A short row (7 entries on the 7-point level, 6-8 on its prolongator's slices) is one trip with its loads
// overlapped, where a 4-deep trip followed by one dependent col -> x chain per remaining entry waited on memory once
// per entry (256^3 Poisson on a B200: level-0 SpMV 0.292 -> 0.259 ms, profiles/r04_sliced_depth.md).
constexpr int SELL_UNROLL = 8;

template <int DEPTH, typename XS, typename V>
__device__ __forceinline__ V sb_sliced_row_sum(const int *cp, const V *vp, int len, const XS &xs) {
    V sum = V(0);
    for (int j = 0; j < len; j += DEPTH) {
        int c[DEPTH];
        V a[DEPTH];
#pragma unroll
        for (int q = 0; q < DEPTH; ++q) {
            const bool in = j + q < len;
            c[q] = in ? sb_ld_stream(cp + (j + q) * 32) : 0;
            a[q] = in ? sb_ld_stream(vp + (j + q) * 32) : V(0);
        }
#pragma unroll
        for (int q = 0; q < DEPTH; ++q)
            if (j + q < len) sum += a[q] * xs.ld(c[q]);
    }
    return sum;
}

// DEPTH: SELL_UNROLL, or 4 in the fused halo kernel, which runs 8 CTAs an SM (32 registers) and would spill at 8
template <int EPI, typename XS, int DEPTH = SELL_UNROLL, typename V>
__device__ __forceinline__ void
spmv_sell_body(int vb, int row_begin, int M, const long long *__restrict__ slice_ptr, const int *__restrict__ col,
               const V *__restrict__ val, const XS xs, const EpiArgsT<V> &e,
               const uint32_t *__restrict__ skip_mask) {
    const int row = row_begin + vb * blockDim.x + threadIdx.x;  // rows [row_begin, M), row_begin % 32 == 0
    const int lane = threadIdx.x & 31;
    const int slice = row >> 5;
    if ((slice << 5) >= M) return;
    const long long base = slice_ptr[slice];
    const int len = (int)((slice_ptr[slice + 1] - base) >> 5);
    const V sum = sb_sliced_row_sum<DEPTH>(col + base + lane, val + base + lane, len, xs);
    if (row < M && !sb_row_skipped(skip_mask, row)) sb_epilogue<EPI>(row, sum, e);
}

template <int EPI, typename V = double>
__global__ void __launch_bounds__(256)
spmv_sell_kernel(int row_begin, int M, const long long *__restrict__ slice_ptr, const int *__restrict__ col,
                 const V *__restrict__ val, const V *__restrict__ x, EpiArgsT<V> e,
                 const uint32_t *__restrict__ skip_mask) {
    spmv_sell_body<EPI>(blockIdx.x, row_begin, M, slice_ptr, col, val, XLocalT<V>{x}, e, skip_mask);
}

// ---------------------------------------------------------------------------------------------
// spmv_sellp: the sliced layout over a row permutation (SELL-C-sigma with C = 32, sigma = 256 = one CTA).  Slot t of
// the grid works on row perm[t]; the rows of a CTA's 256 slots are the 256 consecutive rows of its window, sorted by
// length, so every slice is nearly rectangular whatever the row-length distribution; the row sums go back to row
// order through shared memory, so the epilogue's vector streams are as coalesced as in spmv_sell.  Each row is
// summed by one lane in column order, exactly as in spmv_sell: same result, bit for bit.
// ---------------------------------------------------------------------------------------------
template <int EPI, typename XS, typename V>
__device__ __forceinline__ void
spmv_sellp_body(int vb, int M, const long long *__restrict__ slice_ptr, const int *__restrict__ perm,
                const int *__restrict__ col, const V *__restrict__ val, const XS xs, const EpiArgsT<V> &e) {
    // blockDim.x == 256 == the window; the grid holds exactly ceil(M / 256) CTAs, so every slot exists
    __shared__ V s_sum[256];
    const int slot = vb * 256 + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const int slice = slot >> 5;
    const long long base = slice_ptr[slice];
    const int len = (int)((slice_ptr[slice + 1] - base) >> 5);
    const V sum = sb_sliced_row_sum<SELL_UNROLL>(col + base + lane, val + base + lane, len, xs);
    // back to row order through shared memory: the window's rows are the 256 consecutive rows from vb * 256, each in
    // exactly one slot, so thread t finishes row vb * 256 + t and the epilogue's vector streams stay coalesced
    const int wbase = vb * 256;
    const int row = perm[slot];
    if (row >= 0) s_sum[row - wbase] = sum;
    __syncthreads();
    const int mine = wbase + threadIdx.x;
    if (mine < M) sb_epilogue<EPI>(mine, s_sum[threadIdx.x], e);
}

template <int EPI, typename V = double>
__global__ void __launch_bounds__(256)
spmv_sellp_kernel(int M, const long long *__restrict__ slice_ptr, const int *__restrict__ perm,
                  const int *__restrict__ col, const V *__restrict__ val, const V *__restrict__ x, EpiArgsT<V> e) {
    spmv_sellp_body<EPI>(blockIdx.x, M, slice_ptr, perm, col, val, XLocalT<V>{x}, e);
}

// ---------------------------------------------------------------------------------------------
// spmv_symdiag: symmetric diagonals (mapping 103), one thread per row.  d holds diagonal 0 and the positive offsets
// k of an exactly symmetric operator as dense arrays d_q[M] (q = index of k in s.off); row i's lower entry a_{i,i-k} is
// d_q[i-k].  Row i sums its terms in ascending column order -- lower terms for k descending, d_0[i] x[i], upper terms
// for k ascending -- with the `sum += a * x` chain of sb_sliced_row_sum, so a row sum has the bits of the sliced and
// CSR kernels (a slot the pattern leaves empty holds 0.0 and adds a zero).  Terms outside [0, M) are skipped.
// Loads: d_q[i] is the first touch of its line and stays cached in L2 (.cg) until d_q[i-k], k rows later, reads it
// again as the last use (.cs, evict first).  ND: the kernel's bucket (4, 8, 16 diagonals), s.nd <= ND of them stored.
// ---------------------------------------------------------------------------------------------
template <int ND, int EPI, typename V = double>
__global__ void __launch_bounds__(256)
spmv_symdiag_kernel(int M, const V *__restrict__ d, const SymDiagOffsets s, const V *__restrict__ x,
                    EpiArgsT<V> e) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= M) return;
    const size_t m = (size_t)M;
    // every load of the row in flight before the first use
    V la[ND], lx[ND], ua[ND], ux[ND];
    // (in the reverse of the order the terms are summed: the first multiply-add needs the last load issued, so the
    // compiler has no partial sum to start before every load is in flight)
#pragma unroll
    for (int q = ND - 1; q >= 1; --q) {
        const bool up = q < s.nd && i < M - s.off[q];
        ua[q] = up ? __ldcg(d + q * m + i) : V(0);
        ux[q] = up ? __ldg(x + (i + s.off[q])) : V(0);
    }
    const V a0 = __ldcg(d + i), x0 = __ldg(x + i);
#pragma unroll
    for (int q = 1; q < ND; ++q) {
        const bool lo = q < s.nd && i >= s.off[q];
        la[q] = lo ? __ldcs(d + q * m + (i - s.off[q])) : V(0);
        lx[q] = lo ? __ldg(x + (i - s.off[q])) : V(0);
    }
    // a skipped term is 0.0 * 0.0: adding +0 leaves a non-zero sum as it is, and keeps the chain free of branches
    // (with a branch per term the compiler issues the upper loads only after the lower terms are summed)
    V sum = V(0);
#pragma unroll
    for (int q = ND - 1; q >= 1; --q) sum += la[q] * lx[q];
    sum += a0 * x0;
#pragma unroll
    for (int q = 1; q < ND; ++q) sum += ua[q] * ux[q];
    sb_epilogue<EPI>(i, sum, e);
}

// ---------------------------------------------------------------------------------------------
// boundary rows: rows with entries in other ranks' columns.  8 or 32 lanes per row: local segment
// (recomputed -- these rows are a few percent of the block) + remote segment read from the ghost
// buffer the halo exchange filled (float when the operator's use_double is false:
// matvec_sparse_float, saena_matrix_matvec.cpp:531-538 widens on use).
// ---------------------------------------------------------------------------------------------
template <int LANES, int EPI, typename OffT, typename GhostT>
__device__ __forceinline__ void
spmv_boundary_body(int vb, int n_brows, const int *__restrict__ brow, const OffT *__restrict__ rowptr,
                   const int *__restrict__ col, const double *__restrict__ val,
                   const int *__restrict__ brow_ptr, const int *__restrict__ bcol,
                   const double *__restrict__ bval, const double *__restrict__ x,
                   const GhostT *__restrict__ ghost, const EpiArgs &e) {
    const int gid = vb * blockDim.x + threadIdx.x;
    const int b = gid / LANES, sub = gid % LANES;
    double sum = 0.0;
    int row = -1;
    if (b < n_brows) {
        row = brow[b];
        const OffT s = rowptr[row], t = rowptr[row + 1];
        for (OffT k = s + sub; k < t; k += LANES * VEC_UNROLL) {
            int c[VEC_UNROLL];
            double a[VEC_UNROLL];
#pragma unroll
            for (int q = 0; q < VEC_UNROLL; ++q) {
                const OffT kk = k + q * LANES;
                const bool in = kk < t;
                c[q] = in ? col[kk] : 0;
                a[q] = in ? val[kk] : 0.0;
            }
#pragma unroll
            for (int q = 0; q < VEC_UNROLL; ++q) sum += a[q] * __ldg(x + c[q]);
        }
        const int rs = brow_ptr[b], rt = brow_ptr[b + 1];
        for (int k = rs + sub; k < rt; k += LANES) sum += bval[k] * (double)ghost[bcol[k]];
    }
#pragma unroll
    for (int o = LANES / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (sub == 0 && row >= 0) sb_epilogue<EPI>(row, sum, e);
}

template <int LANES, int EPI, typename OffT, typename GhostT>
__global__ void __launch_bounds__(256)
spmv_boundary_kernel(int n_brows, const int *__restrict__ brow, const OffT *__restrict__ rowptr,
                     const int *__restrict__ col, const double *__restrict__ val,
                     const int *__restrict__ brow_ptr, const int *__restrict__ bcol,
                     const double *__restrict__ bval, const double *__restrict__ x,
                     const GhostT *__restrict__ ghost, const unsigned long long *__restrict__ epoch, int ghost_stride,
                     EpiArgs e) {
    // peer-memory exchange with separate launches (p2p_halo.cu): two landing buffers, the current one follows from
    // the receiving role's application counter; NCCL path: epoch == nullptr, one typed buffer
    if (epoch) ghost += (size_t)(epoch[1] & 1ull) * (size_t)ghost_stride;
    spmv_boundary_body<LANES, EPI, OffT, GhostT>(blockIdx.x, n_brows, brow, rowptr, col, val, brow_ptr, bcol, bval, x,
                                                 ghost, e);
}

// merged mode: ghost values that travelled as float are widened into the tail of x_ext
static __global__ void widen_ghost_kernel(int n, const float *__restrict__ in, double *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (double)in[i];
}

// halo pack: vSend[i] = v[vIndex[i]] (saena_matrix_matvec.cpp:25-26; :463-464 casts to float)
template <typename SendT>
__global__ void halo_pack_kernel(int n, const int *__restrict__ vIndex, const double *__restrict__ v,
                                 SendT *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (SendT)v[vIndex[i]];
}

// ---------------------------------------------------------------------------------------------
// Block SpMV: one pass over the operator for k <= K right-hand sides (saena_b200_solve_pcg_block).  The block is k
// ordinary vectors back to back, column-major: x's column j starts at x + j * ldx (ldx = n_local_cols), every epilogue
// vector's at + j * ld (ld = M).  Each entry's value, column id and row offset is loaded once and applied to the k
// gathered x values; columns j >= k are predicated off, nothing is padded in memory.  Per column every row is summed
// in the order, with the multiply-adds and the epilogue arithmetic, of the single kernel of the same mapping: column j
// of a block application has the bits of the single application to column j.
// ---------------------------------------------------------------------------------------------
template <int EPI, int K>
__device__ __forceinline__ void sb_epilogue_block(int i, long long ld, int k, const double (&ax)[K], const EpiArgs &e) {
#pragma unroll
    for (int j = 0; j < K; ++j)
        if (j < k) sb_epilogue_at<EPI>(i, (long long)i + j * ld, ax[j], e);
}

// sb_sliced_row_sum for K columns: the same trips, loads and per-column `sum += a * x` chain
template <int DEPTH, int K>
__device__ __forceinline__ void sb_sliced_row_sums(const int *cp, const double *vp, int len, const double *x,
                                                   long long ldx, int k, double (&sum)[K]) {
#pragma unroll
    for (int j = 0; j < K; ++j) sum[j] = 0.0;
    for (int t = 0; t < len; t += DEPTH) {
        int c[DEPTH];
        double a[DEPTH];
#pragma unroll
        for (int q = 0; q < DEPTH; ++q) {
            const bool in = t + q < len;
            c[q] = in ? sb_ld_stream(cp + (t + q) * 32) : 0;
            a[q] = in ? sb_ld_stream(vp + (t + q) * 32) : 0.0;
        }
#pragma unroll
        for (int q = 0; q < DEPTH; ++q)
            if (t + q < len) {
#pragma unroll
                for (int j = 0; j < K; ++j)
                    if (j < k) sum[j] += a[q] * __ldg(x + (c[q] + j * ldx));
            }
    }
}

template <int EPI, int K>
__global__ void __launch_bounds__(256)
spmv_sell_block_kernel(int row_begin, int M, int k, const long long *__restrict__ slice_ptr, const int *__restrict__ col,
                       const double *__restrict__ val, const double *__restrict__ x, long long ldx, EpiArgs e,
                       long long ld) {
    const int row = row_begin + blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const int slice = row >> 5;
    if ((slice << 5) >= M) return;
    const long long base = slice_ptr[slice];
    const int len = (int)((slice_ptr[slice + 1] - base) >> 5);
    double sum[K];
    sb_sliced_row_sums<SELL_UNROLL, K>(col + base + lane, val + base + lane, len, x, ldx, k, sum);
    if (row < M) sb_epilogue_block<EPI, K>(row, ld, k, sum, e);
}

template <int EPI, int K>
__global__ void __launch_bounds__(256)
spmv_sellp_block_kernel(int M, int k, const long long *__restrict__ slice_ptr, const int *__restrict__ perm,
                        const int *__restrict__ col, const double *__restrict__ val, const double *__restrict__ x,
                        long long ldx, EpiArgs e, long long ld) {
    __shared__ double s_sum[K][256];
    const int slot = blockIdx.x * 256 + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const int slice = slot >> 5;
    const long long base = slice_ptr[slice];
    const int len = (int)((slice_ptr[slice + 1] - base) >> 5);
    double sum[K];
    sb_sliced_row_sums<SELL_UNROLL, K>(col + base + lane, val + base + lane, len, x, ldx, k, sum);
    const int wbase = blockIdx.x * 256;
    const int row = perm[slot];
    if (row >= 0) {
#pragma unroll
        for (int j = 0; j < K; ++j) s_sum[j][row - wbase] = sum[j];
    }
    __syncthreads();
    const int mine = wbase + threadIdx.x;
    if (mine >= M) return;
#pragma unroll
    for (int j = 0; j < K; ++j) sum[j] = s_sum[j][threadIdx.x];
    sb_epilogue_block<EPI, K>(mine, ld, k, sum, e);
}

// spmv_symdiag_kernel for K columns: the row's stored values are loaded once, then every column is summed with the
// single kernel's chain (skipped terms add 0.0 * 0.0 as there)
template <int ND, int EPI, int K>
__global__ void __launch_bounds__(256)
spmv_symdiag_block_kernel(int M, int k, const double *__restrict__ d, const SymDiagOffsets s,
                          const double *__restrict__ x, long long ldx, EpiArgs e, long long ld) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= M) return;
    const size_t m = (size_t)M;
    double la[ND], ua[ND];
#pragma unroll
    for (int q = ND - 1; q >= 1; --q) {
        const bool up = q < s.nd && i < M - s.off[q];
        ua[q] = up ? __ldcg(d + q * m + i) : 0.0;
    }
    const double a0 = __ldcg(d + i);
#pragma unroll
    for (int q = 1; q < ND; ++q) {
        const bool lo = q < s.nd && i >= s.off[q];
        la[q] = lo ? __ldcs(d + q * m + (i - s.off[q])) : 0.0;
    }
#pragma unroll
    for (int j = 0; j < K; ++j) {
        if (j >= k) break;
        const double *xj = x + j * ldx;
        double lx[ND], ux[ND];
#pragma unroll
        for (int q = ND - 1; q >= 1; --q) ux[q] = (q < s.nd && i < M - s.off[q]) ? __ldg(xj + (i + s.off[q])) : 0.0;
        const double x0 = __ldg(xj + i);
#pragma unroll
        for (int q = 1; q < ND; ++q) lx[q] = (q < s.nd && i >= s.off[q]) ? __ldg(xj + (i - s.off[q])) : 0.0;
        double sum = 0.0;
#pragma unroll
        for (int q = ND - 1; q >= 1; --q) sum += la[q] * lx[q];
        sum += a0 * x0;
#pragma unroll
        for (int q = 1; q < ND; ++q) sum += ua[q] * ux[q];
        sb_epilogue_at<EPI>(i, (long long)i + j * ld, sum, e);
    }
}

// spmv_vec_body for K columns
template <int LANES, int EPI, int K, typename OffT>
__global__ void __launch_bounds__(256)
spmv_vec_block_kernel(int row_begin, int M, int k, const OffT *__restrict__ rowptr, const int *__restrict__ col,
                      const double *__restrict__ val, const double *__restrict__ x, long long ldx, EpiArgs e,
                      long long ld) {
    constexpr int G = 32 / LANES;
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int row0 = row_begin + warp * 32;
    if (row0 >= M) return;
    const int my_row = row0 + lane;
    OffT my_start = 0, my_end = 0;
    if (my_row < M) {
        my_start = rowptr[my_row];
        my_end = rowptr[my_row + 1];
    }
    double mine[K];
#pragma unroll
    for (int j = 0; j < K; ++j) mine[j] = 0.0;
    const int g = lane / LANES;
    const int sub = lane % LANES;
    // (not unrolled, unlike the single kernel: K sums per step, unrolled LANES times, would spill)
#pragma unroll 1
    for (int t = 0; t < LANES; ++t) {
        const int src = t * G + g;
        const OffT start = __shfl_sync(0xffffffffu, my_start, src);
        const OffT end = __shfl_sync(0xffffffffu, my_end, src);
        double sum[K];
#pragma unroll
        for (int j = 0; j < K; ++j) sum[j] = 0.0;
        for (OffT kk0 = start + sub; kk0 < end; kk0 += LANES * VEC_UNROLL) {
            int c[VEC_UNROLL];
            double a[VEC_UNROLL];
#pragma unroll
            for (int q = 0; q < VEC_UNROLL; ++q) {
                const OffT kk = kk0 + q * LANES;
                const bool in = kk < end;
                c[q] = in ? sb_ld_stream(col + kk) : 0;
                a[q] = in ? sb_ld_stream(val + kk) : 0.0;
            }
#pragma unroll
            for (int q = 0; q < VEC_UNROLL; ++q) {
#pragma unroll
                for (int j = 0; j < K; ++j)
                    if (j < k) sum[j] += a[q] * __ldg(x + (c[q] + j * ldx));
            }
        }
#pragma unroll
        for (int j = 0; j < K; ++j) {
#pragma unroll
            for (int o = LANES / 2; o > 0; o >>= 1) sum[j] += __shfl_xor_sync(0xffffffffu, sum[j], o);
            const double v = __shfl_sync(0xffffffffu, sum[j], (lane % G) * LANES);
            if (lane / G == t) mine[j] = v;
        }
    }
    if (my_row < M) sb_epilogue_block<EPI, K>(my_row, ld, k, mine, e);
}

// spmv_rowgroup_body for K columns
template <int TPR, int EPI, int K, typename OffT>
__global__ void __launch_bounds__(256)
spmv_rowgroup_block_kernel(int row_begin, int M, int k, const OffT *__restrict__ rowptr, const int *__restrict__ col,
                           const double *__restrict__ val, const double *__restrict__ x, long long ldx, EpiArgs e,
                           long long ld) {
    constexpr int ROWS = 256 / TPR;
    constexpr int WPR = TPR / 32;
    __shared__ double s_part[K][8];
    const int g = threadIdx.x / TPR, sub = threadIdx.x % TPR;
    const int row = row_begin + blockIdx.x * ROWS + g;
    double sum[K];
#pragma unroll
    for (int j = 0; j < K; ++j) sum[j] = 0.0;
    if (row < M) {
        const OffT start = rowptr[row], end = rowptr[row + 1];
        for (OffT kk0 = start + sub; kk0 < end; kk0 += TPR * VEC_UNROLL) {
            int c[VEC_UNROLL];
            double a[VEC_UNROLL];
#pragma unroll
            for (int q = 0; q < VEC_UNROLL; ++q) {
                const OffT kk = kk0 + q * TPR;
                const bool in = kk < end;
                c[q] = in ? sb_ld_stream(col + kk) : 0;
                a[q] = in ? sb_ld_stream(val + kk) : 0.0;
            }
#pragma unroll
            for (int q = 0; q < VEC_UNROLL; ++q) {
#pragma unroll
                for (int j = 0; j < K; ++j)
                    if (j < k) sum[j] += a[q] * __ldg(x + (c[q] + j * ldx));
            }
        }
    }
#pragma unroll
    for (int j = 0; j < K; ++j) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum[j] += __shfl_xor_sync(0xffffffffu, sum[j], o);
    }
    if (WPR == 1) {
        if (sub == 0 && row < M) sb_epilogue_block<EPI, K>(row, ld, k, sum, e);
    } else {
        if ((threadIdx.x & 31) == 0) {
#pragma unroll
            for (int j = 0; j < K; ++j) s_part[j][threadIdx.x >> 5] = sum[j];
        }
        __syncthreads();
        if (sub == 0 && row < M) {
            double tot[K];
#pragma unroll
            for (int j = 0; j < K; ++j) {
                tot[j] = 0.0;
#pragma unroll
                for (int w = 0; w < WPR; ++w) tot[j] += s_part[j][g * WPR + w];
            }
            sb_epilogue_block<EPI, K>(row, ld, k, tot, e);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// host side: the mappings with one body per row range -- spmv_vec (1..16), spmv_rowgroup (32..256) and the sliced
// layout -- launched alone (operator.cu) or inside the fused halo kernel (fused_halo.cu).  The streaming row blocks
// and the sorted sliced layout have launches of their own.
// ---------------------------------------------------------------------------------------------
// calls f(std::integral_constant<int, MAP>{}) with MAP = mapping; false (nothing called) for any other code
template <typename F>
bool sb_dispatch_mapping(int mapping, F &&f) {
    switch (mapping) {
#define SB_MAP_CASE(MAP)                                                                           \
    case MAP: f(std::integral_constant<int, MAP>{}); return true;
        SB_MAP_CASE(1) SB_MAP_CASE(2) SB_MAP_CASE(4) SB_MAP_CASE(8) SB_MAP_CASE(16)
        SB_MAP_CASE(32) SB_MAP_CASE(64) SB_MAP_CASE(128) SB_MAP_CASE(256) SB_MAP_CASE(SB_MAPPING_SELL)
#undef SB_MAP_CASE
    }
    return false;
}

// 256-thread CTAs over nrows rows: 8 warps x 32 rows (sub-warp, sliced), 256 / mapping rows (row groups)
inline int sb_mapping_blocks(int mapping, int nrows) {
    if (nrows <= 0) return 0;
    const int rows_per_block = (mapping == SB_MAPPING_SELL || mapping < 32) ? 256 : 256 / mapping;
    return (nrows + rows_per_block - 1) / rows_per_block;
}
