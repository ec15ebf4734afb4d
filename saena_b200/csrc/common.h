// common.h -- internal declarations shared by the .cu files of libsaena_b200.so.
// Nothing here is part of the ABI (that is include/saena_b200.h).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "saena_b200.h"

// ---------------------------------------------------------------------------------------------
// error plumbing: every ABI entry point returns int and records a message in the context
// ---------------------------------------------------------------------------------------------
extern thread_local std::string g_sb_init_error;

#define SB_CUDA(call)                                                                              \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            ctx->error = std::string(#call) + ": " + cudaGetErrorString(e_) + " (" + __FILE__ +    \
                         ":" + std::to_string(__LINE__) + ")";                                     \
            return 1;                                                                              \
        }                                                                                          \
    } while (0)

#define SB_FAIL(text)                                                                              \
    do {                                                                                           \
        ctx->error = std::string(text) + " (" + __FILE__ + ":" + std::to_string(__LINE__) + ")";   \
        return 1;                                                                                  \
    } while (0)

#define SB_TRY(expr)                                                                               \
    do {                                                                                           \
        int rc_ = (expr);                                                                          \
        if (rc_) return rc_;                                                                       \
    } while (0)

// ---------------------------------------------------------------------------------------------
// SpMV epilogues: what one thread does with (A x)_i.  Fusing them into the SpMV is what makes a
// smoother sweep / residual / prolong+correct a single pass over the operator.
// ---------------------------------------------------------------------------------------------
enum EpiKind {
    EPI_PLAIN = 0,       // out = Ax                                  (matvec)
    EPI_RESIDUAL = 1,    // out = Ax - rhs                            (saena_matrix.tpp:16-23)
    EPI_CHEB_FIRST = 2,  // d = c1*invd*(rhs-Ax); dout=d; out=u+d      (saena_matrix.cpp:1099-1109)
    EPI_CHEB_NEXT = 3,   // d = c1*din + c2*invd*(rhs-Ax); out=u+d     (saena_matrix.cpp:1111-1130)
    EPI_JACOBI = 4,      // out = u - (Ax-rhs)*(invd*omega)            (saena_matrix.cpp:1061-1069)
    EPI_SUB = 5,         // out = u - Ax                               (prolong + correct, solve.cpp:1325,1360)
    EPI_COUNT = 6
};

template <typename V>
struct EpiArgsT {
    const V *rhs;
    const V *inv_diag;
    const V *d_in;
    V *d_out;
    const V *u_in;
    V *out;
    V c1, c2;
};
using EpiArgs = EpiArgsT<double>;
// the FP32 preconditioner's (saena_b200_set_precond_precision): float vectors, the constants computed in double on the
// host and rounded to float at launch
using EpiArgs32 = EpiArgsT<float>;

// ---------------------------------------------------------------------------------------------
// device-side operator
// ---------------------------------------------------------------------------------------------
struct HaloPeer {
    int peer;
    int offset;  // element offset into the packed send / ghost buffer
    int count;
};

// Peer-memory halo (csrc/halo_sync.cuh, fused_halo.cu, p2p_halo.cu): one slice of the packed send order, where it
// lands in the receiving rank's landing area (IPC-mapped, doubles, TWO buffers selected by the parity of the
// application count) and the counter the last pack CTA raises there.
struct HaloSeg {
    long long start;              // first packed element of this receiver's slice
    long long count;
    double *dst;                  // slice of buffer 0 in the receiver's landing area
    long long dst_stride;         // elements between the receiver's two buffers (= its recvSize)
    unsigned long long *arrived;  // flag in the RECEIVER's arena: "values of application k have landed" (= k + 1)
};

// Device-side state of one operator's hand-shake.  All counters are monotonic (application counts), nothing is ever
// reset, so a launch carries no host-side state and replays from a CUDA graph.
struct HaloSyncDev {
    unsigned long long *epoch = nullptr;  // [2] applications completed by the pack role / by the receiving role
    unsigned int *tickets = nullptr;      // [2] last-CTA detection of the two roles
    HaloSeg *segs = nullptr;                         // [sends.size()]
    unsigned long long **wait_consumed = nullptr;    // [sends.size()] my arena: receiver r has consumed application k
    unsigned long long **wait_arrived = nullptr;     // [recvs.size()] my arena: sender s's application k has landed
    unsigned long long **signal_consumed = nullptr;  // [recvs.size()] the senders' arenas
};

// sliced layout (32-slot slices, column-major inside a slice, padded per slice to its longest row), built on the
// device from the CSR arrays.  perm: slot -> row (-1: no row) of the sorted layout; nullptr: slot = row.
struct SlicedLayout {
    long long *ptr = nullptr;  // [n_slices+1] element offsets
    int *perm = nullptr;
    int *col = nullptr;
    double *val = nullptr;
    float *val32 = nullptr;  // FP32 copy of val (FP32 preconditioner, sb_f32_sync); shares ptr, perm and col
};

// the stored diagonals of mapping 103: off[0] = 0, then the positive offsets ascending (kernel argument, by value)
static const int SYMDIAG_MAX = 16;
static const int SYMDIAG_RULE_MAX = 4;   // the most stored diagonals sb_choose_mapping picks mapping 103 for
struct SymDiagOffsets {
    int nd = 0;
    int off[SYMDIAG_MAX] = {};
};

struct DevOperator {
    bool present = false;
    int kind = 0, level = 0;
    int M = 0, n_local_cols = 0, col_offset = 0;
    int64_t nnz_local = 0, nnz_remote = 0;
    bool use_double = true;
    bool wide_offsets = false;  // 64-bit row offsets (nnz_local >= 2^31)
    // saena_matrix::use_dense (saena_b200_set_operator_dense): with use_double false the reference's dense
    // product casts the whole input vector to float; x_round holds that rounded copy during an application
    bool use_dense = false;
    double *x_round = nullptr;  // [n_local_cols], allocated when use_dense && !use_double

    // local block: CSR, column ids LOCAL (global - col_offset)
    void *rowptr = nullptr;  // int32[M+1] or int64[M+1]
    int *col = nullptr;
    double *val = nullptr;
    float *val32 = nullptr;  // FP32 copy of val while a mapping 1..256 is in use at precision 32 (sb_f32_sync)

    // row blocks of the streaming kernel: rows [blk_row[b], blk_row[b+1]) hold <= STREAM_TILE nnz
    int *blk_row = nullptr;
    int n_blk = 0;

    // sliced layout in row order (mapping 100) for short regular rows
    SlicedLayout sell;
    int64_t sell_padded_est = 0;    // stored entries incl. padding the sliced layout would have (computed at upload)
    bool sell_only = false;         // the CSR col/val were released once the sliced copy existed (no other mapping)

    // sliced layout over a row permutation (mapping 101): inside every window of 256 consecutive rows (one CTA) the
    // rows are sorted by length, longest first, so that the 32 rows of a slice have nearly the same length and the
    // padding of irregular operators (unstructured matrices, smoothed prolongators) all but disappears.  Operators
    // without a halo only.  Never chosen by the heuristic: set_mapping / autotune.
    SlicedLayout sellp;

    // symmetric diagonals (mapping 103): an exactly symmetric square operator whose entries lie on a few diagonals,
    // stored as dense double[sdiag.nd][M] arrays of diagonal 0 and the positive offsets only -- no column ids.  Row i
    // reads its lower entry a_{i,i-k} as d_k[i-k] (= a_{i-k,i}, same bits).  One rank, no halo, not merged.
    // sdiag_n: -1 not probed yet, 0 not eligible, > 0 the stored diagonals (sdiag.off).  sdiag_val: null unless built.
    SymDiagOffsets sdiag;
    int sdiag_n = -1;
    double *sdiag_val = nullptr;
    float *sdiag_val32 = nullptr;  // FP32 copy of sdiag_val (sb_f32_sync)

    // remote block re-sorted by row at upload: boundary rows only
    // interior rows = the contiguous range [int_lo, int_hi) (multiples of 32) that holds no row with
    // remote entries: for a slab partition the rows touching ghosts sit at the two ends of the
    // block.  The overlapped kernel runs on that range only; everything outside is a "boundary
    // row" finished after the halo arrives -- nothing is computed twice.
    int int_lo = 0, int_hi = 0;
    int n_brows = 0;
    int *brow = nullptr;       // [n_brows] local row id, ascending
    int *brow_ptr = nullptr;   // [n_brows+1]
    int *bcol = nullptr;       // [nnz_remote] index into the ghost buffer
    double *bval = nullptr;    // [nnz_remote]
    uint32_t *brow_mask = nullptr;  // bit i set <=> row i has remote entries (local kernel skips its epilogue)

    // merged mode: when most rows touch ghost columns (deep coarse levels: every row couples to
    // every rank) the local/remote split degenerates.  The operator is then stored ONCE over the
    // extended column space [local columns | ghost columns] and applied to x_ext = [x | ghosts]
    // after the exchange, with the ordinary kernels.
    bool merged = false;
    double *x_ext = nullptr;  // [n_local_cols + recvSize]
    int *rowmid = nullptr;    // merged, 32-bit offsets: where the ghost columns of each row start (rows are [local | ghost])
    double *partial = nullptr;  // [M] local-column sums kept across the wait of the fused kernel (fused_halo.cu)

    // halo plan
    int vIndexSize = 0, recvSize = 0;
    int *vIndex = nullptr;
    void *send_buf = nullptr;  // double[vIndexSize] or float[vIndexSize]
    void *ghost_buf = nullptr; // double[recvSize] or float[recvSize]
    std::vector<HaloPeer> sends, recvs;

    // peer-memory path (set by saena_b200_p2p_import; the NCCL path stays as the fallback).  p2p: ghost values are
    // stored by the senders into ghost_d over NVLink.  fused: the whole application is ONE kernel (fused_halo.cu);
    // otherwise separate launches (p2p_halo.cu: pack kernel on the comm stream, interior kernel, wait, boundary
    // kernel, release).  Both speak the same hand-shake on the same flags and landing buffers, so the choice is free
    // per operator, per rank and per application.
    bool p2p = false;
    bool fused = false;
    float tune_ms[2] = {0.f, 0.f};                // saena_b200_autotune_halo: fused / separate launches
    double *ghost_d = nullptr;                    // landing area in the arena, 2 x recvSize doubles (double-buffered)
    size_t ghost_arena_off = 0;                   // NCCL path: where this operator's typed ghost area / x_ext starts
    size_t ghost_d_off = 0;
    int op_id = 0;                                // level * 3 + kind (fault reports)
    HaloSyncDev hs;

    // kernel mapping: the canonical code of saena_b200_set_mapping that sb_choose_mapping settled on (1..16 lanes
    // per row, 32..256 threads per row, -1..-32 streaming row blocks with -mapping lanes per row in the reduce
    // phase, SB_MAPPING_SELL, SB_MAPPING_SELLP; 0 until the operator is prepared)
    int mapping = 0;
    int forced_mapping = 0;   // the code requested by set_mapping / the autotune (0: the nnz/row rule)

    double avg_nnz_row() const { return M ? double(nnz_local + nnz_remote) / M : 0.0; }
};

struct RepartPlan {
    std::vector<saena_b200_block> send, recv;
    bool identity() const { return send.empty() && recv.empty(); }
};

struct DevLevel {
    DevOperator A, P, R;
    // the operator of an ABI kind (SAENA_B200_KIND_*); any kind other than A or P is R
    DevOperator &op(int kind) { return kind == SAENA_B200_KIND_A ? A : (kind == SAENA_B200_KIND_P ? P : R); }
    const DevOperator &op(int kind) const { return const_cast<DevLevel *>(this)->op(kind); }
    double *inv_diag = nullptr;
    double *inv_sq_diag = nullptr;  // inv_sq_diag_orig, only for scale=true hierarchies
    double eig_max = 0.0;
    int M = 0;             // A.M
    int M_coarse_old = 0;  // Ac.M_old
    int M_coarse = 0;      // Ac.M
    RepartPlan repart;
    bool aux_set = false;
    // A is applied as R_{l-1} (A_{l-1} (P_{l-1} x)) instead of streaming the stored Galerkin product
    // (sb_apply_level_A; chosen by saena_b200_autotune_mapping or saena_b200_set_level_route, reset by finalize)
    bool route = false;
    float route_ms[2] = {0.f, 0.f};  // autotune: median ms of a Chebyshev sweep on the stored A / on the route (0: not timed)

    // work vectors (Grid::allocate_mem + the smoother's temp1/temp2)
    double *u[2] = {nullptr, nullptr};  // ping-pong iterate; u[cur] is current
    int cur = 0;
    double *d = nullptr;         // Chebyshev direction (temp2)
    double *res = nullptr;       // residual (Grid::res)
    double *rhs = nullptr;       // this level's right-hand side (parent's res_coarse after repart); level 0: external
    double *xfer_old = nullptr;  // coarse vector in the old partition (Ac.M_old), used when repart is not identity

    // the same work vectors for a block of up to ctx->blk_cap columns, column-major (column j at + j * M, xfer_old's
    // at + j * M_coarse_old); allocated by sb_block_reserve on the first block call, bcur is their ping-pong parity
    double *bu[2] = {nullptr, nullptr};
    int bcur = 0;
    double *bd = nullptr, *bres = nullptr, *brhs = nullptr, *bxfer_old = nullptr;

    // FP32 preconditioner (precision 32, sb_f32_sync): the work vectors above in float, with the same ping-pong parity
    // cur; level 0's rhs32 is the converted PCG residual.  inv_diag32: inv_diag rounded to float.
    float *u32[2] = {nullptr, nullptr};
    float *d32 = nullptr, *res32 = nullptr, *rhs32 = nullptr, *inv_diag32 = nullptr;
};

// a level's work vectors in one precision: what the templated smoother and V-cycle of solve.cu run on
template <typename V>
struct LevelVecs {
    V **u;
    V *d, *res, *rhs;
    const V *inv_diag;
};
inline LevelVecs<double> sb_level_vecs(DevLevel &lv, double) { return {lv.u, lv.d, lv.res, lv.rhs, lv.inv_diag}; }
inline LevelVecs<float> sb_level_vecs(DevLevel &lv, float) {
    return {lv.u32, lv.d32, lv.res32, lv.rhs32, lv.inv_diag32};
}

// A V-cycle from a zero iterate is the same launch sequence every time (same buffers, same
// per-level Chebyshev constants): it is captured once per (rhs, smoother, pre, post) into a CUDA
// graph and replayed -- the coarse levels are launch-latency-bound, ~90 launches per V-cycle.
struct VcycleGraph {
    const void *rhs;
    int smoother, pre, post;
    cudaGraphExec_t exec;
    int64_t launches;
    std::vector<int> cur_after;  // each level's ping-pong parity when the V-cycle ends
    int k = 0;                   // 0: the single V-cycle; 1..SB_BLOCK_MAX: the block V-cycle on k columns
    int bits = 64;               // 64: the FP64 V-cycle; 32: the FP32 one (k = 0)
    // exec == nullptr: a multi-rank configuration that has run eagerly once and is captured at its next use
};

struct saena_b200_ctx {
    int device = 0, rank = 0, nranks = 1;
    bool detached = false;  // saena_b200_init_detached: a rank's share with no peer (compute-only profiling)
    std::string error;
    cudaStream_t stream = nullptr;  // compute
    cudaStream_t comm_stream = nullptr;
    cudaEvent_t ev_packed = nullptr, ev_halo = nullptr, ev_t0 = nullptr, ev_t1 = nullptr;
    void *nccl_comm = nullptr;
    int sm_count = 148;
    std::vector<DevLevel> levels;
    bool finalized = false;
    bool use_graphs = true;
    bool nvtx = false;               // SAENA_B200_NVTX=1
    bool use_graphs_multi = true;   // capture with nranks > 1 too (SAENA_B200_GRAPH_MULTI=0 turns it off)
    int64_t graph_replays = 0;
    std::vector<VcycleGraph> graphs;
    bool scale = false;  // saena_object::scale
    int fused_restrict_levels = 0;  // levels [0, n) run residual + restriction as ONE scatter kernel (fused_restrict.cu); 0: off
    // fused kernel on merged operators: local columns summed before the wait, ghost columns after.  Opt-in
    // (SAENA_B200_MERGED_SPLIT=1): measured at N=2 on 256^3 it LOSES (levels 3-4: 1.52 / 0.67 ms per V-cycle against
    // 1.38 / 0.61 -- the second reduction and the second walk over the row offsets cost more than the ~10 us of
    // exchange they hide); kept for the latency-bound many-rank case
    bool merged_split = false;
    // operator upload: merged layout from this fraction of rows with remote entries.  0.25 in round 1; measured in
    // round 2: the rows outside the clean run take the boundary-row kernel at ~1/3 of the interior mapping's rate, so
    // already 12 % of such rows cost level 1 of the 512^3 hierarchy on 8 GPUs a third of its time (1.459 ms per sweep
    // against 1.078 ms for the same rows on one GPU), while a merged operator only gives up the ~30 us of overlap;
    // 256^3 on 4 GPUs: levels 1-2 -3 % / -6 % at 0.08 (profiles/r02_bench_n4_merge_above_0.08.json)
    double merge_above = 0.08;
    int apply_mode = 0;  // measurement only: 0 full, 1 local kernels only (no exchange), 2 pack + exchange only
    int64_t launches = 0;

    // coarsest dense factor
    int coarse_n = 0;
    double *coarse_A = nullptr;     // [n*n] row-major
    double *coarse_Ainv = nullptr;  // [n*n] row-major
    double *coarse_tmp = nullptr;   // [2n]
    bool coarsest_cg = false;       // direct_solver == "CG": solve_coarsest_CG instead of the dense factor
    double *ccg_res = nullptr, *ccg_dir = nullptr, *ccg_mv = nullptr;
    int ccg_cap = 0;

    // reductions
    double *red_partials = nullptr;  // [RED_MAX_BLOCKS * 4]
    unsigned int *red_counter = nullptr;
    double *scalars = nullptr;       // device scalars of the Krylov loop
    double *scalars_host = nullptr;  // pinned mirror

    // PCG vectors (level-0 size)
    double *pcg_r = nullptr, *pcg_p = nullptr, *pcg_h = nullptr, *pcg_u = nullptr, *pcg_rhs = nullptr;
    int pcg_cap = 0;

    // hook staging (host <-> device copies of the per-operator hooks)
    double *stage[4] = {nullptr, nullptr, nullptr, nullptr};
    size_t stage_cap[4] = {0, 0, 0, 0};

    // halo arena (nranks > 1): flags + every operator's ghost area in ONE allocation, so that one
    // IPC handle per rank maps everything a neighbour needs to write into
    char *arena = nullptr;
    size_t arena_bytes = 0;
    std::vector<void *> peer_arena;  // [nranks] IPC mappings of the peers' arenas (nullptr: not opened)
    bool p2p_ready = false;
    // bounded waits (halo_sync.cuh): a spin that outlives halo_timeout_ns records what it waited for in fault_dev and
    // every later wait drains at once; the ABI call that ran into it returns non-zero (the reference's convention is
    // print + MPI_Abort, src/saena_object_solve.cpp:1012-1013; the adaptor maps the status to that).
    unsigned long long *fault_dev = nullptr;   // = (unsigned long long *)(scalars + S_COUNT): code, wanted, seen, spare
    unsigned long long halo_timeout_ns = 5000000000ull;   // SAENA_B200_HALO_TIMEOUT_MS
    double sync_timeout_s = 180.0;             // host-side watchdog of every blocking wait (SAENA_B200_SYNC_TIMEOUT_S)
    bool faulted = false;                      // sticky until saena_b200_clear_fault
    bool fused_default = true;  // p2p_import switches eligible operators to the fused kernel (SAENA_B200_HALO_FUSED=0: no)

    double *tune_dev = nullptr;   // [32] scratch of the collective mapping autotune (all-reduce MAX of candidate times)

    // the two fine-level intermediates of a route level (P_{l-1} x, A_{l-1} P_{l-1} x); allocated while a level is
    // on the route or being timed for it
    double *route_t = nullptr, *route_s = nullptr;
    int route_cap = 0;

    // FP32 preconditioner (saena_b200_set_precond_precision): 64 (default) or 32.  At 32 the FP32 copies of the values
    // in use, inv_diag32 and the levels' float work vectors exist; f32_stale: some call since their last build may
    // have changed values, layouts, the route or the coarsest solver (set by sb_invalidate_graphs), so sb_f32_sync
    // builds them again before the next FP32 use.  route32_*: the route's intermediates in float.
    int precond_bits = 64;
    bool f32_stale = false;
    float *route32_t = nullptr, *route32_s = nullptr;

    // L2 flush buffer for the timing loops
    void *flush_buf = nullptr;
    size_t flush_bytes = 0;

    // host-clock ms of the last saena_b200_update_values, by phase (refresh.cu: UPDATE_PHASES)
    double update_ms[5] = {0.0, 0.0, 0.0, 0.0, 0.0};

    // block solve (sb_block_reserve): work vectors for up to blk_cap columns -- the levels' (DevLevel::bu ...), the
    // PCG's and the route's -- and reduction state of its own: per column a row of RED_MAX_BLOCKS partials and a
    // counter, and the scalars as blk_scal[slot * SB_BLOCK_MAX + column] (slots as ctx->scalars', S_COUNT of them)
    int blk_cap = 0;
    size_t blk_route_cap = 0;  // elements of each route intermediate (columns x the routed fine level's rows)
    double *blk_r = nullptr, *blk_p = nullptr, *blk_h = nullptr, *blk_u = nullptr, *blk_rhs = nullptr;
    double *blk_route_t = nullptr, *blk_route_s = nullptr;
    double *blk_partials = nullptr;   // [SB_BLOCK_MAX * RED_MAX_BLOCKS]
    unsigned int *blk_counter = nullptr;  // [SB_BLOCK_MAX]
    double *blk_scal = nullptr;       // [S_COUNT * SB_BLOCK_MAX]
    double *blk_scal_host = nullptr;  // pinned mirror
    int *blk_active = nullptr;        // [SB_BLOCK_MAX] 1: the column still iterates (the PCG updates skip the others)
    int *blk_active_host = nullptr;   // pinned mirror

    // GMRES (saena_b200_solve_gmres, sb_gmres_reserve): one allocation of 2 * gm_cap + 2 level-0 vectors at stride
    // gm_ld -- the basis v_0 .. v_cap, the preconditioned vectors z_0 .. z_{cap-1} and the preconditioner's input t --
    // grown to the largest restart so far; and the reduction state of the Arnoldi kernels (krylov.cu), its own
    int gm_cap = 0;
    long long gm_ld = 0;
    double *gm_vec = nullptr;
    double *gm_partials = nullptr;      // [(SB_GMRES_MAX + 2) * RED_MAX_BLOCKS]
    unsigned int *gm_counter = nullptr;
    double *gm_scal = nullptr;          // krylov.cu: the reductions' sums and the Hessenberg column
    double *gm_scal_host = nullptr;     // pinned mirror
};

// scalar slots
enum { S_RHO_RES = 0, S_PDOTH = 1, S_RR = 2, S_BETA_NUM = 3, S_TMP = 4,
       S_C_RR = 8, S_C_DEN = 9, S_C_RRNEW = 10,  // coarsest-level CG (must not clobber the outer loop's)
       S_AGREE = 11,                             // number of ranks whose halo exchange timed out (sb_agree_fault)
       S_COUNT = 16,
       S_FAULT_WORDS = 4 };  // the halo fault record follows the scalars: one copy brings both to the host

static const int SB_MAPPING_SELL = 100;   // forced_mapping / set_mapping code of the sliced layout
static const int SB_MAPPING_SELLP = 101;  // ... of the sliced layout with rows sorted by length inside 256-row windows
static const int SB_MAPPING_SYMDIAG = 103;  // ... of the symmetric diagonals (DevOperator::sdiag)
static const int STREAM_TILE = 2048;      // nnz per row block of the streaming kernel (16 KB of products)
static const int STREAM_THREADS = 256;
static const int RED_MAX_BLOCKS = 1184;   // 148 SMs x 8
static const int SB_BLOCK_MAX = 8;        // right-hand sides of one block solve
static const int SB_GMRES_MAX = 64;       // largest GMRES restart length

// ---------------------------------------------------------------------------------------------
// NVTX ranges (SAENA_B200_NVTX=1): the stages the reference's PROFILE_PCG / PROFILE_VCYCLE builds time
// (/root/reference/include/saena_object.h:24-26, :434-440 -- Rtransfer, Ptransfer, smooth, coarsest, residual,
// repart, dots, level-0 matvec), as named ranges for a timeline profiler.  Off by default: no call is made.
// ---------------------------------------------------------------------------------------------
struct SbRange {
    bool on;
    SbRange(const saena_b200_ctx *ctx, const char *name, int level = -1);
    ~SbRange();
};

// ---- operator.cu
int sb_upload_operator(saena_b200_ctx *ctx, const saena_b200_operator_desc *d);
int sb_upload_band_operator(saena_b200_ctx *ctx, int level, int n, int half_bandwidth, int sliced_only);
void sb_free_operator(DevOperator &op);
void sb_choose_mapping(saena_b200_ctx *ctx, DevOperator &op);
int sb_prepare_operator(saena_b200_ctx *ctx, DevOperator &op);
void sb_drop_unused_layouts(DevOperator &op);
void sb_sellp_layout(int M, const int64_t *rowptr, int *perm, long long *slice_ptr);
// (re)writes the entries of an existing sliced layout of op from its CSR arrays (slice offsets and perm in place)
int sb_fill_sliced(saena_b200_ctx *ctx, const DevOperator &op, SlicedLayout &s);
// host only: the stored diagonals of mapping 103 for an operator of M rows, nnz entries, `padded_est` sliced entries
// and these distinct offsets col - row; 0 when the layout does not apply (stored: SYMDIAG_MAX ints)
int sb_symdiag_plan(int M, int n_offsets, const int *offsets, int64_t nnz, int64_t padded_est, int *stored);
// after new values on the same pattern (saena_b200_update_values): an operator on mapping 103 gets its diagonals
// filled again; when the new values are not symmetric it moves to the sliced layout
int sb_refresh_symdiag(saena_b200_ctx *ctx, DevOperator &op);
// w-style application of an operator with a fused epilogue; x is the local input vector.
int sb_apply(saena_b200_ctx *ctx, DevOperator &op, const double *x, int epi, const EpiArgs &args);
// ---- spmv_f32.cu
// the same on the operator's FP32 copy (precision 32: one rank, no halo, not merged, no streaming row blocks)
int sb_apply(saena_b200_ctx *ctx, DevOperator &op, const float *x, int epi, const EpiArgs32 &args);
// dst = (float)src / (double)src, and the FP32 copies' cast
int sb_convert(saena_b200_ctx *ctx, size_t n, const double *src, float *dst);
int sb_convert(saena_b200_ctx *ctx, size_t n, const float *src, double *dst);
// ---- spmv_block.cu
// sb_apply on k column-major vectors: x's column j at x + j * n_local_cols, the epilogue's at + j * M (inv_diag shared)
int sb_apply_block(saena_b200_ctx *ctx, DevOperator &op, int k, const double *x, int epi, const EpiArgs &args);
// algorithmic bytes of one application with vb-byte values and vector elements (8: FP64, 4: FP32 preconditioner)
int64_t sb_operator_bytes(const DevOperator &op, int vb = 8);

// ---- nccl_comm.cu
int sb_nccl_unique_id(void *out, std::string &err);
int sb_nccl_init(saena_b200_ctx *ctx, const void *id);
void sb_nccl_destroy(saena_b200_ctx *ctx);
int sb_halo_exchange(saena_b200_ctx *ctx, DevOperator &op, cudaStream_t s);
int sb_allreduce_sum(saena_b200_ctx *ctx, double *dev_vals, int count, cudaStream_t s);
int sb_allreduce_max(saena_b200_ctx *ctx, double *dev_vals, int count, cudaStream_t s);
// moves blocks of `src` to the peers' `dst`; forward: send plan -> recv plan, backward: reversed
int sb_repart(saena_b200_ctx *ctx, const RepartPlan &plan, bool backward, const double *src, double *dst,
              cudaStream_t s);

// ---- p2p_halo.cu
int sb_arena_build(saena_b200_ctx *ctx);     // at finalize: allocate the arena, point ghost buffers into it
void sb_arena_free(saena_b200_ctx *ctx);
// separate-launch form of the peer-memory exchange (same hand-shake as the fused kernel)
int sb_p2p_pack(saena_b200_ctx *ctx, DevOperator &op, const double *x, cudaStream_t s);   // wait consumed, pack, raise arrived
int sb_p2p_wait_arrived(saena_b200_ctx *ctx, DevOperator &op, cudaStream_t s);            // 1 CTA spins (bounded)
int sb_p2p_gather_ghosts(saena_b200_ctx *ctx, DevOperator &op, double *dst, cudaStream_t s);  // current buffer -> dst
int sb_p2p_release(saena_b200_ctx *ctx, DevOperator &op, cudaStream_t s);                 // raise consumed, advance epoch

// ---- fused_halo.cu
bool sb_fused_eligible(const DevOperator &op);
int sb_apply_fused(saena_b200_ctx *ctx, DevOperator &op, const double *x, int epi, const EpiArgs &args);

// ---- api.cu
int sb_sync_stream(saena_b200_ctx *ctx, cudaStream_t s);   // cudaStreamSynchronize with a watchdog
int sb_check_fault(saena_b200_ctx *ctx);                   // non-zero (and ctx->error set) once a halo wait has timed out
// collective end of a solver call: all ranks return the same status (one all-reduce of the fault flags), so no rank
// leaves the sequence of collective calls while the others go on
int sb_agree_fault(saena_b200_ctx *ctx);
// the coarsest level's dense factor from its global COO (host LU + inverse, kept on the device); n in 1..4096
int sb_coarsest_factor(saena_b200_ctx *ctx, int n, int64_t nnz, const int32_t *row, const int32_t *col, const double *val);
// probes every level on the route again and takes off the route each one whose stored A_l no longer matches R A P
int sb_recheck_routes(saena_b200_ctx *ctx);

// ---- refresh.cu
// saena_b200_update_values on values already on the device (checks first, then writes)
int sb_update_values(saena_b200_ctx *ctx, const double *val_dev, int64_t nnz, int max_eig_iter, unsigned long long seed,
                     double *dropped_out, int dropped_cap);

// ---- fused_restrict.cu
int sb_residual_restrict_fused(saena_b200_ctx *ctx, int l, const double *u, const double *rhs, double *res_coarse);

// ---- vector_ops.cu
int sb_dot(saena_b200_ctx *ctx, const double *a, const double *b, int n, int slot);           // scalars[slot] = <a,b> (global)
int sb_cheb_first_zero(saena_b200_ctx *ctx, int n, const double *rhs, const double *inv_diag, double c, double *d,
                       double *u);                                                          // u = d = c*invd*rhs
int sb_pcg_update(saena_b200_ctx *ctx, int n, double *u, double *r, const double *p, const double *h);  // + scalars[S_RR]
int sb_pcg_p_update(saena_b200_ctx *ctx, int n, double *p, const double *rho);
int sb_cg_p_update(saena_b200_ctx *ctx, int n, double *p, const double *r, int num_slot, int den_slot);
int sb_negate_copy(saena_b200_ctx *ctx, int n, const double *src, double *dst);              // dst = -src
int sb_fill_zero(saena_b200_ctx *ctx, double *p, size_t n);
// float forms (FP32 preconditioner)
int sb_cheb_first_zero(saena_b200_ctx *ctx, int n, const float *rhs, const float *inv_diag, float c, float *d, float *u);
int sb_negate_copy(saena_b200_ctx *ctx, int n, const float *src, float *dst);
int sb_fill_zero(saena_b200_ctx *ctx, float *p, size_t n);
int sb_scale_vector(saena_b200_ctx *ctx, int n, double *v, const double *w);                   // v *= w (scale_vector)
int sb_coarsest_apply(saena_b200_ctx *ctx, const double *rhs, double *u);
int sb_coarsest_cg(saena_b200_ctx *ctx, const double *rhs, double *u);  // u: initial guess in, solution out
int sb_read_scalars(saena_b200_ctx *ctx);  // device scalars -> scalars_host (synchronises the stream)
// Block forms on k column-major columns of n rows (column j at + j * n).  Each column goes through the single kernel's
// arithmetic: the reductions use the same CTA count and summation tree per column, with the block's own partials and
// counters, and write blk_scal[slot * SB_BLOCK_MAX + j].  The PCG updates take per-column alpha / beta from blk_scal
// and leave the columns whose blk_active entry is 0 as they are.
int sb_dot_block(saena_b200_ctx *ctx, const double *a, const double *b, int n, int k, int slot);
int sb_pcg_update_block(saena_b200_ctx *ctx, int n, int k, double *u, double *r, const double *p, const double *h);
int sb_pcg_p_update_block(saena_b200_ctx *ctx, int n, int k, double *p, const double *rho);
int sb_cheb_first_zero_block(saena_b200_ctx *ctx, int n, int k, const double *rhs, const double *inv_diag, double c,
                             double *d, double *u);
int sb_negate_copy_block(saena_b200_ctx *ctx, int n, int k, const double *src, double *dst);
int sb_scale_vector_block(saena_b200_ctx *ctx, int n, int k, double *v, const double *w);
int sb_read_block_scalars(saena_b200_ctx *ctx);  // blk_scal -> blk_scal_host (synchronises the stream)

// ---- krylov.cu (GMRES's Arnoldi process; every pass on level-0 vectors of n rows at stride ld)
int sb_gmres_state(saena_b200_ctx *ctx);        // the reduction state, allocated once
void sb_gmres_state_free(saena_b200_ctx *ctx);
void sb_gmres_free(saena_b200_ctx *ctx);        // api.cu: the workspace and the reduction state
// w = A z_j orthogonalised in place against the nv vectors V (CGS2); the Hessenberg column h_0 .. h_{nv-1}, ||w||
// after and ||w|| before the orthogonalisation land in the device scalars (sb_gmres_read, sb_gmres_column_host)
int sb_gmres_orthogonalize(saena_b200_ctx *ctx, int n, long long ld, const double *V, int nv, double *w);
int sb_gmres_norm2(saena_b200_ctx *ctx, int n, const double *w);   // <w, w> (sb_gmres_norm2_host after a read)
int sb_gmres_normalize(saena_b200_ctx *ctx, int n, double *v, double h, double *t);   // v /= h; t = v
int sb_gmres_update(saena_b200_ctx *ctx, int n, long long ld, const double *Z, int k, const double *y, double *x);
int sb_gmres_read(saena_b200_ctx *ctx);         // device scalars -> pinned mirror (synchronises the stream)
double sb_gmres_norm2_host(const saena_b200_ctx *ctx);
const double *sb_gmres_h1_host(const saena_b200_ctx *ctx);      // first pass's dots, |w|^2 after them
const double *sb_gmres_h2_host(const saena_b200_ctx *ctx);      // second pass's dots, |w'|^2 after them
const double *sb_gmres_column_host(const saena_b200_ctx *ctx);  // h1 + h2, ||w''||, ||w||

// ---- lanczos.cu
// out = uniform(-1, 1) from a counter-based generator on the global row index (row_offset + i)
int sb_fill_random(saena_b200_ctx *ctx, int n, long long row_offset, unsigned long long seed, double *out);
int sb_find_eig(saena_b200_ctx *ctx, int level, int max_iter, const double *start_dev, unsigned long long seed,
                double *eig_out, int *iters_out);

// ---- solve.cu
// Each with an FP64 and an FP32 form (the FP32 preconditioner): one template, the same steps on the level's work
// vectors of that precision (sb_level_vecs), the operators through the sb_apply of that precision.
// level l's operator with a fused epilogue: the stored A_l, or on a route level R_{l-1} A_{l-1} P_{l-1}
int sb_apply_level_A(saena_b200_ctx *ctx, int l, const double *x, int epi, const EpiArgs &args);
int sb_apply_level_A(saena_b200_ctx *ctx, int l, const float *x, int epi, const EpiArgs32 &args);
int64_t sb_level_A_bytes(const saena_b200_ctx *ctx, int l, int vb = 8);  // algorithmic bytes of what sb_apply_level_A streams
int sb_smooth(saena_b200_ctx *ctx, int l, int smoother, int iters, const double *rhs, bool u_is_zero);
int sb_smooth(saena_b200_ctx *ctx, int l, int smoother, int iters, const float *rhs, bool u_is_zero);
int sb_vcycle(saena_b200_ctx *ctx, int l, int smoother, int pre, int post, const double *rhs, bool u_is_zero);
int sb_vcycle(saena_b200_ctx *ctx, int l, int smoother, int pre, int post, const float *rhs, bool u_is_zero);
// level-0 V-cycle from a zero iterate, replayed from a CUDA graph when nothing in it needs the host (graphs keyed by
// precision too)
int sb_vcycle_from_zero(saena_b200_ctx *ctx, int smoother, int pre, int post, const double *rhs);
int sb_vcycle_from_zero(saena_b200_ctx *ctx, int smoother, int pre, int post, const float *rhs);
void sb_invalidate_graphs(saena_b200_ctx *ctx);
// the block forms on k columns of the levels' block buffers (DevLevel::bu[bcur] is the iterate)
int sb_apply_level_A_block(saena_b200_ctx *ctx, int l, int k, const double *x, int epi, const EpiArgs &args);
int sb_smooth_block(saena_b200_ctx *ctx, int l, int k, int smoother, int iters, const double *rhs, bool u_is_zero);
int sb_vcycle_block(saena_b200_ctx *ctx, int l, int k, int smoother, int pre, int post, const double *rhs,
                    bool u_is_zero);
// the level-0 block V-cycle from a zero iterate, replayed from a CUDA graph like sb_vcycle_from_zero's
int sb_vcycle_block_from_zero(saena_b200_ctx *ctx, int k, int smoother, int pre, int post, const double *rhs);

// ---- api.cu (block solve)
// block buffers for k columns (grown to the largest k so far, and to the routed levels; growing drops every captured
// block V-cycle); a failed allocation leaves no block buffer and the context usable for single solves
int sb_block_reserve(saena_b200_ctx *ctx, int k);
void sb_block_free(saena_b200_ctx *ctx);

// ---- api.cu (FP32 preconditioner)
// Before every FP32 use: when stale, checks the refusal rules again, builds every FP32 copy anew from the FP64 data
// (values of the layout in use, inv_diag, work vectors, the route's intermediates) and drops the captured FP32 V-cycles.
// The one place the copies are written.  On a refusal or a failed allocation the context goes back to 64.
int sb_f32_sync(saena_b200_ctx *ctx);
void sb_f32_free(saena_b200_ctx *ctx);
