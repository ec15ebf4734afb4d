/*
 * saena_b200.h -- C ABI of the B200-native AMG solve phase (the drop-in boundary).
 *
 * The reference (paralab/Saena) has no FFI layer: its boundary is the C++ pImpl
 * API of include/saena.hpp whose solve methods forward into saena_object
 * (/root/reference/src/saena.cpp:745-799).  This header is what a replacement
 * of those forwarders binds (see INTEGRATION.md for the adaptor): the finished
 * hierarchy that saena_object::setup left in `grids` is uploaded once, then
 * solve_pCG / solve / the per-operator hooks run on the GPU.
 *
 * Conventions
 *  - plain C: pointers + sizes, no C++/torch types.  Host pointers unless a
 *    parameter is named *_dev.
 *  - every function returns 0 on success, non-zero on failure and never calls
 *    exit(); saena_b200_last_error() gives the message.  (The reference's
 *    convention is print-and-terminate, SURVEY.md 8b; the adaptor maps
 *    non-zero to that.)
 *  - one context per process/GPU (= one MPI rank of the reference).  With
 *    nranks > 1 all calls that touch a distributed level are collective and
 *    must be made in the same order on every rank (as the reference's are).
 *  - FP64 values, int32 row/column indices (Saena's value_t / index_t,
 *    include/data_struct.h:36-38); nnz counts are 64-bit (nnz_t).
 *  - there is no CPU fallback: if no CUDA device is usable, init fails.
 */
#ifndef SAENA_B200_H
#define SAENA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct saena_b200_ctx saena_b200_ctx;

#define SAENA_B200_NCCL_ID_BYTES 128

enum { SAENA_B200_KIND_A = 0, SAENA_B200_KIND_P = 1, SAENA_B200_KIND_R = 2 };
enum { SAENA_B200_JACOBI = 0, SAENA_B200_CHEBYSHEV = 1 };

/* ---- lifecycle ------------------------------------------------------------------------ */

/* Rank 0 creates the NCCL id and shares the 128 bytes with the other ranks by any means (the
 * reference's ranks share MPI_COMM_WORLD, experiments/Poisson.cpp:18-22). */
int saena_b200_nccl_unique_id(void *id_out);

/* nccl_id may be NULL when nranks == 1 (no communicator is created). */
int saena_b200_init(saena_b200_ctx **ctx_out, int device_id, int rank, int nranks, const void *nccl_id);
/* Profiling aid: rank `rank`'s share of an nranks-way partition on one GPU with no peer behind it
 * (no NCCL, no peer memory).  Uploads and finalize work as usual; any operation that needs a peer
 * fails loudly; saena_b200_time_matvec_compute_only times the compute side of the distributed
 * kernels on that share -- the way to put the fused halo kernel under ncu, which cannot follow a
 * multi-rank command. */
int saena_b200_init_detached(saena_b200_ctx **ctx_out, int device_id, int rank, int nranks);
int saena_b200_destroy(saena_b200_ctx *ctx);
const char *saena_b200_last_error(const saena_b200_ctx *ctx); /* ctx may be NULL: error of a failed init */

/* ---- hierarchy upload (once per setup) ---------------------------------------------------
 * The descriptor carries the arrays of one operator exactly as the reference's setup built
 * them: saena_matrix::set_off_on_diagonal (src/saena_matrix_setup.cpp:793-1098),
 * prolong_matrix::findLocalRemote (src/prolong_matrix.cpp:18-378),
 * restrict_matrix::transposeP (src/restrict_matrix.cpp:229-494); field names are the
 * reference's member names (include/saena_matrix.h:105-149).                              */
typedef struct saena_b200_operator_desc {
    int32_t kind;                    /* SAENA_B200_KIND_* */
    int32_t level;                   /* grids[level] */
    int32_t M;                       /* local rows */
    int32_t n_local_cols;            /* length of the local input vector */
    int32_t col_offset;              /* split[rank] of the column partition: kernels index v - col_offset */
    int32_t use_double;              /* 0: ghost values travel as float (matvec_sparse_float) */
    int64_t nnz_local;
    const int32_t *nnzPerRow_local;  /* [M] */
    const int32_t *col_local;        /* [nnz_local] GLOBAL ids, row-major */
    const double *val_local;         /* [nnz_local] */
    int64_t nnz_remote;
    int32_t col_remote_size;         /* == recvSize */
    const int32_t *row_remote;       /* [nnz_remote] local row, column-major grouped by owner */
    const double *val_remote;        /* [nnz_remote] */
    const int32_t *nnzPerCol_remote; /* [col_remote_size] */
    int32_t vIndexSize;
    const int32_t *vIndex;           /* [vIndexSize] local ids whose values are sent */
    int32_t numSendProc;
    const int32_t *sendProcRank;     /* [numSendProc] */
    const int32_t *sendProcCount;    /* [numSendProc] */
    const int32_t *vdispls;          /* [nranks] start of each receiver's slice in the send buffer */
    int32_t numRecvProc;
    const int32_t *recvProcRank;     /* [numRecvProc] */
    const int32_t *recvProcCount;    /* [numRecvProc] */
    const int32_t *rdispls;          /* [nranks] start of each sender's slice in the ghost buffer */
} saena_b200_operator_desc;

int saena_b200_upload_operator(saena_b200_ctx *ctx, const saena_b200_operator_desc *desc);

/* Measurement input (one rank): the A operator of `level` generated on the device with the pattern
 * and values of saena::band_matrix (src/aux_functions2.cpp:1296-1381, experiments/banded.cpp) --
 * row i = columns [i-b, i+b] inside [0, n), value 1/(i+j+1).  BASELINE.json configs[3] is 50 M
 * rows x 129 entries = 77 GB with 64-bit row offsets, more than a host upload can feed a bench run;
 * the arrays are the ones saena_b200_upload_operator would build from the same matrix.
 * sliced_only != 0: once finalize has built the sliced (32-row slice, column-major) copy the CSR
 * entries are released -- CSR + sliced copy of the full-size case would be 156 GB -- and the
 * operator keeps that one mapping. */
int saena_b200_upload_band_operator(saena_b200_ctx *ctx, int level, int n, int half_bandwidth, int sliced_only);

/* (peer, offset, count) of Grid::repart_u's plan (src/grid.cpp:3-163): offset is into the
 * old-partition vector for sends and into the new-partition vector for receives. */
typedef struct saena_b200_block {
    int32_t peer, offset, count;
} saena_b200_block;

/* Per-level data next to A_l: inv_diag and eig_max_of_invdiagXA (saena_matrix.h:151,183) and
 * the plan that moves R's output (Ac.M_old entries) onto the coarse grid's partition (Ac.M). */
int saena_b200_upload_level_aux(saena_b200_ctx *ctx, int level, const double *inv_diag, double eig_max,
                                int M_coarse_old, int M_coarse, int n_send, const saena_b200_block *send,
                                int n_recv, const saena_b200_block *recv);

/* Only for a hierarchy set up with scale=true (saena::amg::set_scale, saena::matrix::assemble(true)):
 * D^-1/2 of each level's unscaled operator (saena_matrix::inv_sq_diag_orig).  The V-cycle scales
 * the restricted residual and the coarse correction with the coarse level's vector
 * (src/saena_object_solve.cpp:1245-1247, :1264-1266) and the solvers scale the final u with level
 * 0's (:2709-2711).  Uploading it for level 0 switches the scaled path on. */
int saena_b200_upload_level_scale(saena_b200_ctx *ctx, int level, const double *inv_sq_diag_orig);

/* Coarsest operator as global COO (what setup_SuperLU passes on, saena_object_solve.cpp:282-308).
 * It is LU-factored on the host once and kept on the device as a dense factor; the rank that
 * owns the coarsest level's rows applies it (the others pass n = 0). */
int saena_b200_upload_coarsest(saena_b200_ctx *ctx, int n, int64_t nnz, const int32_t *row, const int32_t *col,
                               const double *val);

/* saena_matrix::use_dense of an uploaded A operator (include/saena_matrix.h:191; set by the setup when
 * switch_to_dense is on, the coarse operator's density exceeds dense_thre and Mbig <= dense_sz_thre,
 * src/saena_object_setup2.cpp:328-329).  The reference then applies the operator through
 * saena_matrix_dense::matvec (include/saena_matrix.tpp:5-7, src/saena_matrix_dense.cpp:181-340): the same
 * matrix and the same product, except that with use_double == 0 the WHOLE input vector is cast to float
 * before it is multiplied -- the rank's own part too (:281-282), where matvec_sparse_float only casts the
 * ghost values.  The device keeps applying the operator from its sparse arrays (such levels hold at most
 * dense_sz_thre = 5000 rows: latency-bound either way) and reproduces that cast: the input is rounded
 * through float on the way into the kernel.  Call after saena_b200_upload_operator, before finalize. */
int saena_b200_set_operator_dense(saena_b200_ctx *ctx, int level, int kind, int use_dense);

/* saena_object::direct_solver (include/saena_object.h:165): 0 = the direct solve (default, "SuperLU"
 * in the reference, the dense factor here), 1 = solve_coarsest_CG (src/saena_object_solve.cpp:14-114). */
int saena_b200_set_coarsest_solver(saena_b200_ctx *ctx, int use_cg);

/* The preconditioner's V-cycle is replayed from a CUDA graph when it contains no host-side
 * decision: captured on first use on one rank; on several ranks the first V-cycle of a
 * configuration runs eagerly and the second is captured -- halo flags, peer stores, the comm
 * stream's fork/join and the ncclSend/ncclRecv of Grid::repart_u included (environment
 * SAENA_B200_GRAPH_MULTI=0 keeps several ranks eager).  0 switches graphs off. */
int saena_b200_set_graphs(saena_b200_ctx *ctx, int on);
/* V-cycles replayed from a graph by this context since init */
int64_t saena_b200_graph_replays(const saena_b200_ctx *ctx);

/* Seal the hierarchy: allocates the per-level work vectors (Grid::allocate_mem, grid.cpp:165-172)
 * and picks each operator's kernel mapping from its nnz/row. */
int saena_b200_finalize(saena_b200_ctx *ctx);

/* ---- peer-memory halo (nranks > 1, all ranks on one NVLink/NVSwitch node) ----------------------
 * After finalize every rank exports a small blob (IPC handle of its halo arena + where each
 * sender's values land), the host all-gathers the blobs over whatever channel it has
 * (MPI_Allgather in the adaptor, torch.distributed in bench.py) and every rank imports the
 * concatenation (rank order, `blob_bytes` each); no rank applies an operator before all have
 * returned from the import (barrier).  From then on the ghost values of the distributed
 * SpMV are stored by the sender straight into the receiver's memory over NVLink, and the whole
 * distributed operator application -- pack + peer stores, interior rows, rows that wait for the
 * ghost values, fused epilogue -- is ONE kernel (csrc/fused_halo.cu; what matvec_sparse,
 * src/saena_matrix_matvec.cpp:9-113, does with MPI_Isend/Irecv/Waitany around two loops).
 * saena_b200_p2p_enable selects the transport: 2 = that fused kernel (default after the import),
 * 1 = peer stores with separate launches (pack kernel on a comm stream, interior kernel, wait
 * kernel, boundary kernel, release kernel), 0 = ncclSend/ncclRecv (what runs without the import).
 * 1 and 2 are two forms of ONE hand-shake (csrc/halo_sync.cuh: monotonic counters, two landing
 * buffers per operator), so they may be mixed freely per operator, per rank and per application;
 * only the switch between 0 and non-zero is collective.  p2p_export with buf == NULL only reports
 * the size.
 *
 * Failure detection.  Every device-side wait of the exchange is bounded (SAENA_B200_HALO_TIMEOUT_MS,
 * default 5000): a wait that runs out records what it was waiting for, every later wait of the
 * context drains at once, and the ABI call in which it happened returns non-zero with the operator,
 * counter and values in saena_b200_last_error -- each rank on its own clock, never a hang.  Every
 * blocking host wait is bounded too (SAENA_B200_SYNC_TIMEOUT_S, default 180: a peer process that
 * died inside a collective).  The reference's convention for a failed rank is print + MPI_Abort
 * (src/saena_object_solve.cpp:1012-1013); the adaptor maps the status to that.  After a timed-out
 * exchange the counters of the ranks are out of step: saena_b200_clear_fault (every rank) followed
 * by saena_b200_p2p_enable(ctx, 0) continues over NCCL, a new export/import re-arms peer memory. */
int saena_b200_p2p_export(saena_b200_ctx *ctx, void *buf, int64_t cap, int64_t *size_out);
int saena_b200_p2p_import(saena_b200_ctx *ctx, const void *blobs, int64_t blob_bytes);
int saena_b200_p2p_enable(saena_b200_ctx *ctx, int on);
int saena_b200_fault_status(saena_b200_ctx *ctx);  /* 0: no wait of this context has timed out */
int saena_b200_clear_fault(saena_b200_ctx *ctx);
/* deadlines: device-side halo waits in ms (< 0: unchanged), blocking host waits in s (<= 0: unbounded) */
int saena_b200_set_timeouts(saena_b200_ctx *ctx, double halo_timeout_ms, double sync_timeout_s);
/* Measures both peer-memory paths on every operator of the uploaded hierarchy (reps back-to-back
 * applications each, times summed over the ranks) and keeps the faster one per operator.
 * Collective; call after p2p_import.  saena_b200_halo_choice reports the outcome for one operator
 * (1 fused kernel, 0 separate launches / NCCL, -1 no such operator) and this rank's two timings. */
int saena_b200_autotune_halo(saena_b200_ctx *ctx, int reps);
int saena_b200_halo_choice(const saena_b200_ctx *ctx, int level, int kind, float *ms_fused, float *ms_unfused);

/* ---- next to the solve path (SURVEY.md 8f #1): the Chebyshev bound on the device ---------------
 * saena_object::find_eig (src/saena_object.cpp:572-590 -> include/lamlan_saena.h:13-79): largest
 * eigenvalue of D^-1/2 A D^-1/2 by Lanczos (<= max_iter steps, 20 in the reference, full
 * re-orthogonalisation, stop at a 1e-8 relative change of the Ritz value), times 1.0001.  Runs on
 * the uploaded operator of `level` with the solve's own SpMV (distributed when nranks > 1; collective).
 * start: optional host start vector (this rank's rows; the reference draws uniform(-1,1) from
 * std::random_device), NULL = a seeded generator on the global row index.  store != 0 installs the
 * result as the level's bound (eig_max_of_invdiagXA). */
int saena_b200_find_eig(saena_b200_ctx *ctx, int level, int max_iter, const double *start, uint64_t seed, int store,
                        double *eig_out, int *iters_out);

/* ---- next to the solve path (SURVEY.md 8f #4): new values on the same pattern, without a new setup ----------------
 * For a user who solves many systems with one matrix pattern (time steps, Newton steps, coefficient sweeps).  One rank.
 * val_local: new values of level 0's A in the UPLOADED order -- row-major, the nnzPerRow_local / col_local given at
 * upload, nnz_local entries.  The aggregates, P, R, every stored pattern, the kernel mappings, row blocks and the
 * autotune's choices are kept; the values are recomputed:
 *   1. level 0's A takes the values;
 *   2. for l = 0 .. L-1, C = R_l (A_l P_l) on the device (the SpGEMM below) is mapped onto A_{l+1}'s stored pattern with
 *      the setup's filter rule (saena_object::filter): a stored entry takes C's value, an off-diagonal entry of C
 *      outside the pattern is lumped into its row's diagonal, a diagonal below 1e-14 in magnitude (or one C lacks) is 1;
 *      a stored off-diagonal entry that C lacks is an error ("not a Galerkin product of the level above").  With the
 *      uploaded values this reproduces the setup's own A_{l+1};
 *   3. every level's inv_diag = 1 / diag(A_l) and eig_max = find_eig(l, max_eig_iter, NULL, seed, store = 1);
 *   4. the sliced copies of the operators' entries (mappings 100 / 101) and the coarsest dense factor are rebuilt;
 *   5. captured V-cycles are dropped, and a level on the route (saena_b200_set_level_route) stays there only if
 *      R A P still matches its stored operator to the route's tolerance (saena_b200_get_level_route reports it).
 * dropped_out (optional, dropped_cap entries): per level, the lumped entries' share ||C - C|pattern||_F / ||C||_F --
 * how far the frozen pattern has drifted from what a new setup would keep; dropped_out[0] = 0.
 * Refused, with the hierarchy untouched: several ranks (the coarse product of a row-partitioned level needs the other
 * ranks' rows of P), a scaled hierarchy, a context that is not finalized, nnz_local != level 0's, an operator uploaded
 * sliced_only (its CSR values were released), a new level-0 diagonal that is missing or below 1e-14 in magnitude.
 * A failure after writing has begun (a coarse pattern that is not a Galerkin product, a CUDA error) leaves the
 * context un-finalized: every solver and hook refuses until the hierarchy is uploaded again.
 * The _dev variant takes the values in device memory (complete before the call).
 * saena_b200_update_values_times: host-clock ms of the last update's phases -- products, pattern map (with the
 * diagonals), sliced layouts, eigenvalue bounds, coarsest factor (cap <= 5 entries). */
int saena_b200_update_values(saena_b200_ctx *ctx, const double *val_local, int64_t nnz_local, int max_eig_iter,
                             uint64_t seed, double *dropped_out, int dropped_cap);
int saena_b200_update_values_dev(saena_b200_ctx *ctx, const double *val_local_dev, int64_t nnz_local,
                                 int max_eig_iter, uint64_t seed, double *dropped_out, int dropped_cap);
int saena_b200_update_values_times(const saena_b200_ctx *ctx, double *ms_out, int cap);

/* ---- next to the solve path (SURVEY.md 8f #3): the Galerkin product's SpGEMM on the device ----------
 * C = A B for CSR operands (64-bit row offsets, int32 columns, FP64 values), all pointers DEVICE pointers, work on
 * the default stream.  What saena_object::triple_mat_mult (src/saena_object_setup2.cpp:361) computes as R (A P)
 * through the matmat machinery of src/saena_object_setup_matmat.cpp:27-1160 (innermost product: MKL's
 * mkl_dcsrmultcsr, :214-218).  Two calls: symbolic fills c_rowptr[M + 1] and returns nnz(C); the caller allocates
 * c_col / c_val of that size and calls numeric, which writes every row with ascending columns.  A is M x K, B is
 * K x N.  Row-wise Gustavson with per-row accumulators chosen by row size (csrc/spgemm.cu).  No context is needed;
 * errors are reported through saena_b200_last_error(NULL). */
int saena_b200_spgemm_symbolic(int M, int K, int N, const int64_t *a_rowptr, const int32_t *a_col,
                               const int64_t *b_rowptr, const int32_t *b_col, int64_t *c_rowptr, int64_t *nnz_c);
int saena_b200_spgemm_numeric(int M, int K, int N, const int64_t *a_rowptr, const int32_t *a_col, const double *a_val,
                              const int64_t *b_rowptr, const int32_t *b_col, const double *b_val,
                              const int64_t *c_rowptr, int32_t *c_col, double *c_val);

/* ---- solvers -----------------------------------------------------------------------------
 * rhs / u are this rank's block (grids[0].A->M entries).  u is overwritten (zero initial
 * guess, as the reference does: saena_object_solve.cpp:2482).  `iters` receives the count
 * the reference prints ("stopped at iteration", i+1).  hist[0] = ||r0||, hist[k] = ||r_k||.  */
int saena_b200_solve_pcg(saena_b200_ctx *ctx, const double *rhs, double *u, int max_iter, double tol,
                         int smoother, int pre, int post, int *iters, double *hist, int hist_cap,
                         int *hist_len);                                      /* saena_object::solve_pCG */
int saena_b200_solve_vcycle(saena_b200_ctx *ctx, const double *rhs, double *u, int max_iter, double tol,
                            int smoother, int pre, int post, int *iters, double *hist, int hist_cap,
                            int *hist_len);                                   /* saena_object::solve */
int saena_b200_solve_cg(saena_b200_ctx *ctx, const double *rhs, double *u, int max_iter, double tol, int *iters,
                        double *hist, int hist_cap, int *hist_len);           /* saena_object::solve_CG */
/* saena_object::solve_smoother (src/saena_object_solve.cpp:2017-2117): `pre` smoother sweeps per iteration on
 * level 0, nothing else; `post` is unused, as in the reference */
int saena_b200_solve_smoother(saena_b200_ctx *ctx, const double *rhs, double *u, int max_iter, double tol,
                              int smoother, int pre, int post, int *iters, double *hist, int hist_cap,
                              int *hist_len);

/* Same solve with rhs / u already resident in device memory (no host copies). */
int saena_b200_solve_pcg_dev(saena_b200_ctx *ctx, const double *rhs_dev, double *u_dev, int max_iter, double tol,
                             int smoother, int pre, int post, int *iters, double *hist, int hist_cap,
                             int *hist_len);

/* ---- flexible GMRES: nonsymmetric operators, one rank -----------------------------------------------------------
 * Right-preconditioned restarted flexible GMRES(restart) (Saad's FGMRES) with the AMG V-cycle as the preconditioner.
 * For an operator that is not symmetric positive definite, where solve_pcg's CG does not apply: convection-diffusion,
 * a Newton Jacobian with an upwinded term, a Helmholtz-type operator in general form.  The conventions of solve_pcg:
 * zero initial guess, r = A u - rhs, the stop test ||r|| < tol * ||r0|| with r0 = -rhs, the direct solve alone on a
 * one-level hierarchy (iters = 1, hist = {||r0||, ||r||}), and u scaled with level 0's inv_sq_diag_orig at the end on
 * a scaled hierarchy.
 *   Cycle.  v_0 = r / ||r||; inner iteration j: z_j = M^-1 v_j (the V-cycle from a zero iterate, FP32 while
 *   saena_b200_set_precond_precision is 32, as for solve_pcg), w = A z_j, w orthogonalised against v_0 .. v_j by
 *   classical Gram-Schmidt applied twice (h_{i,j} = the sum of both passes' coefficients), h_{j+1,j} = ||w||,
 *   v_{j+1} = w / h_{j+1,j}.  Z = [z_0 ..] is kept next to V, so the preconditioner may change between applications
 *   (the FP32 V-cycle); with the FP64 one this is plain right-preconditioned GMRES.  The small least-squares problem
 *   is solved on the host by Givens rotations; its residual estimate |g_{j+1}| is hist's entry for the iteration.  A
 *   cycle ends when that estimate is below tol * ||r0||, after `restart` inner iterations, at max_iter inner iterations
 *   in all, or at a happy breakdown (h_{j+1,j} = 0 or <= 1e-300 * ||w|| before the orthogonalisation).  Then u -= Z y
 *   (y from the rotated triangle; a zero pivot contributes nothing), the true residual is computed, and the solve
 *   stops if it meets the test or max_iter is reached, else restarts from it.
 *   Outputs.  iters = inner iterations run; hist[0] = ||r0||, hist[k] = the residual estimate after inner iteration k,
 *   so hist_len = iters + 1 (a restart adds no entry).  A zero rhs returns u = 0, iters = 0, hist_len = 1,
 *   hist[0] = 0.  A NaN stops the solve at once: a NaN ||r0|| returns u = 0, iters = 0, hist = {NaN}; a NaN estimate
 *   is its iteration's hist entry and u keeps the iterate of the last finished cycle.
 *   Workspace.  2 * restart + 2 vectors of level 0's length (V, Z and the preconditioner's input), allocated at the
 *   first call with a larger restart than before and freed by finalize and destroy; growing it drops nothing else.
 *   A failed allocation returns non-zero and leaves the context usable for every other solver.
 *   Refused (non-zero, the hierarchy untouched): restart outside 1..64, max_iter < 1, several ranks or a detached share,
 *   a context that is not finalized.
 * Every reduction runs in a fixed order with partials and counters of its own: a repeated solve gives the same bits,
 * with graphs on or off (the V-cycle is replayed from its graph; the Arnoldi step is not captured). */
int saena_b200_solve_gmres(saena_b200_ctx *ctx, const double *rhs, double *u, int restart, int max_iter, double tol,
                           int smoother, int pre, int post, int *iters, double *hist, int hist_cap, int *hist_len);
/* the same with rhs / u in device memory (complete before the call) */
int saena_b200_solve_gmres_dev(saena_b200_ctx *ctx, const double *rhs_dev, double *u_dev, int restart, int max_iter,
                               double tol, int smoother, int pre, int post, int *iters, double *hist, int hist_cap,
                               int *hist_len);
/* Test hook: one orthogonalisation step of the solve's kernels on host vectors.  V: nv (0..64) vectors of n entries
 * back to back; w (n) is replaced by w'' = w' - V h2, where w' = w - V h1.  h1[0..nv) = V^T w with h1[nv] = <w, w>;
 * h2[0..nv) = V^T w' with h2[nv] = <w', w'>; col[0..nv) = h1 + h2, col[nv] = ||w''||, col[nv + 1] = ||w||.  Needs an
 * initialised context only (no hierarchy). */
int saena_b200_gmres_orthogonalize(saena_b200_ctx *ctx, int n, int nv, const double *V, double *w, double *h1,
                                   double *h2, double *col);

/* ---- per-operator hooks (saena::matrix::matvec and the parity tests) --------------------- */
int saena_b200_matvec(saena_b200_ctx *ctx, int level, int kind, const double *v, double *w);
int saena_b200_residual(saena_b200_ctx *ctx, int level, const double *u, const double *rhs, double *res);
int saena_b200_smooth(saena_b200_ctx *ctx, int level, int smoother, int iters, double *u, const double *rhs);
int saena_b200_vcycle(saena_b200_ctx *ctx, int level, int smoother, int pre, int post, double *u,
                      const double *rhs);
int saena_b200_coarsest_solve(saena_b200_ctx *ctx, const double *rhs, double *u);
int saena_b200_dot(saena_b200_ctx *ctx, const double *a, const double *b, int n, double *out);

/* ---- block solve: 1 <= k <= 8 right-hand sides on one hierarchy, one rank --------------------------------------------
 * Every vector argument is a block of k ordinary vectors back to back (column-major): column j starts at
 * base + j * ld, ld = the level's rows (grids[0].A->M for the solve), or the operator's local columns for an operator's
 * input.  Each operator is streamed once for all k columns.  Column j gives exactly -- to the bit -- what the single
 * call gives for column j: for the solve the same iteration count, residual history and u; columns are independent (a
 * zero or NaN column changes no other column).  Every call returns non-zero, and leaves the hierarchy as it was, for
 * k outside 1..8, a context of several ranks (a detached share included) or one not finalized.  The work vectors for k
 * columns (about 2 x the single solve's per column) are allocated at the first call with a larger k than before; an
 * allocation that fails returns non-zero and the context stays usable for single solves. */
/* saena_b200_solve_pcg on k columns: iters[k], hist[k * hist_cap] (column j's history at hist + j * hist_cap),
 * hist_len[k] */
int saena_b200_solve_pcg_block(saena_b200_ctx *ctx, int k, const double *rhs, double *u, int max_iter, double tol,
                               int smoother, int pre, int post, int *iters, double *hist, int hist_cap,
                               int *hist_len);
/* the same with rhs / u in device memory */
int saena_b200_solve_pcg_block_dev(saena_b200_ctx *ctx, int k, const double *rhs_dev, double *u_dev, int max_iter,
                                   double tol, int smoother, int pre, int post, int *iters, double *hist,
                                   int hist_cap, int *hist_len);
/* saena_b200_matvec / _residual / _smooth / _vcycle on k columns */
int saena_b200_matvec_block(saena_b200_ctx *ctx, int level, int kind, int k, const double *v, double *w);
int saena_b200_residual_block(saena_b200_ctx *ctx, int level, int k, const double *u, const double *rhs, double *res);
int saena_b200_smooth_block(saena_b200_ctx *ctx, int level, int smoother, int iters, int k, double *u,
                            const double *rhs);
int saena_b200_vcycle_block(saena_b200_ctx *ctx, int level, int smoother, int pre, int post, int k, double *u,
                            const double *rhs);

/* ---- measurement ---------------------------------------------------------------------------
 * Device-resident timing loops for bench.py: `reps` applications of one operator / smoother
 * sweep, each launch bracketed by CUDA events on the launching stream; returns the median
 * milliseconds per launch.  KIND_A of a level on the route (saena_b200_set_level_route) times the route.  While the
 * preconditioner precision is 32 (saena_b200_set_precond_precision) both time the FP32 kernels the V-cycle runs. */
int saena_b200_time_matvec(saena_b200_ctx *ctx, int level, int kind, int reps, int flush_l2, float *ms_out);
int saena_b200_time_smooth_sweep(saena_b200_ctx *ctx, int level, int smoother, int reps, int flush_l2,
                                 float *ms_out);
/* N > 1 (collective): the same operator application timed three ways -- complete (exchange
 * overlapped with the interior rows), local kernels alone, pack + exchange alone -- so that
 * hidden = 1 - (full - local) / halo can be reported.  Like saena_b200_time_matvec, KIND_A times what the solve
 * applies: the route on a level that takes it (saena_b200_set_level_route). */
int saena_b200_time_matvec_parts(saena_b200_ctx *ctx, int level, int kind, int reps, float *full_ms,
                                 float *local_ms, float *halo_ms);
/* CUDA-event stopwatch on the context's compute stream (the stream every kernel of this library
 * is launched on): start records an event, stop records a second one, waits for it and returns
 * the device time between them. */
/* ms per application of one operator's compute side only (no pack, no flags, no exchange; ghost values
 * as they lie): fused != 0 through the fused halo kernel, else the separate interior + boundary kernels */
int saena_b200_time_matvec_compute_only(saena_b200_ctx *ctx, int level, int kind, int fused, int reps, int do_flush,
                                        float *ms_out);
/* Measurement behind a design decision (one rank): the V-cycle's residual + restriction on `level` as the solve
 * path's two kernels (res = A u - rhs written, then R res) against ONE kernel that scatters every fine residual
 * through its row of P with FP64 atomics and never writes res (csrc/fused_restrict.cu).  Median ms of `reps`
 * launches each and the relative 2-norm difference of the two coarse vectors. */
int saena_b200_time_residual_restrict(saena_b200_ctx *ctx, int level, const double *u, const double *rhs, int reps,
                                      float *ms_two_kernels, float *ms_fused, double *rel_diff);
/* Opt-in: levels [0, levels) of the V-cycle run residual + restriction as that one scatter kernel where the level is
 * eligible (no halo, A on the sliced layout); 0 (default) keeps the two kernels.  Measured: profiles/r02_fused_restrict.md. */
int saena_b200_set_fused_restrict(saena_b200_ctx *ctx, int levels);
int saena_b200_timer_start(saena_b200_ctx *ctx);
/* ms per V-cycle entered at `level` from a zero iterate (reps back-to-back, eager, collective over
 * the ranks); the difference between consecutive levels is one level's cost inside a solve.  While the preconditioner
 * precision is 32 (saena_b200_set_precond_precision) it times the FP32 V-cycle, which is what the solve runs. */
int saena_b200_time_vcycle(saena_b200_ctx *ctx, int level, int smoother, int pre, int post, int reps, float *ms_out);
int saena_b200_timer_stop(saena_b200_ctx *ctx, float *ms_out);
/* median ms of one GMRES orthogonalisation step with nv (1..64) basis vectors of level 0's length: the three CGS2
 * passes and the normalisation, on seeded unit vectors in the solve's workspace (one rank) */
int saena_b200_time_gmres_step(saena_b200_ctx *ctx, int nv, int reps, float *ms_out);
/* kernels launched by this context since init (bench.py's gpu_launches) */
int64_t saena_b200_launch_count(const saena_b200_ctx *ctx);
/* Force one operator's SpMV row mapping (tuning / profiling / tests): 0 = heuristic from nnz/row;
 * 1..16 = that many lanes per row, 32 rows per warp; 32..256 = that many threads per row, one row
 * per thread group; -1..-32 = streaming row blocks with that many lanes per row in the reduce
 * phase; 100 = sliced layout (32-row slices, column-major, one lane per row); 101 = the sliced
 * layout over rows sorted by length inside 256-row windows (irregular rows: the slices' padding all
 * but disappears; operators without a halo only, otherwise the heuristic's choice is kept); 103 = symmetric
 * diagonals (an exactly symmetric square operator on at most 32 diagonals, one rank, no halo: diagonal 0 and the
 * positive offsets as dense arrays, no column ids; the heuristic picks it for such an operator with at most 4 stored
 * diagonals and at least the sliced layout's row count; on an operator that is not eligible the heuristic's choice is
 * kept). */
int saena_b200_set_mapping(saena_b200_ctx *ctx, int level, int kind, int mapping);
/* The same, taking effect at the next saena_b200_finalize (no layout is built for the mapping that
 * is being replaced: matters for an operator that fills half the HBM). */
int saena_b200_set_mapping_deferred(saena_b200_ctx *ctx, int level, int kind, int mapping);
/* Host-only half of mapping 101 (no device needed; what the layout build calls): for row offsets rowptr[M + 1], the
 * slot -> row permutation perm[ceil(M / 256) * 256] (rows of every 256-row window sorted by length, longest first,
 * stable; -1 where the last window runs past M) and slice_ptr[ceil(M / 256) * 8 + 1], the element offset of every
 * 32-slot slice (32 x its longest row). */
int saena_b200_sellp_layout(int M, const int64_t *rowptr, int32_t *perm, long long *slice_ptr);
/* Host only: the rule behind mapping 103 (symmetric diagonals).  For an operator of M rows and nnz entries whose
 * distinct offsets col - row are offsets[n_offsets] and whose sliced layout would store padded_est entries: the number
 * of stored diagonals, written to stored[] (offset 0, then the positive offsets ascending; at most 16), or 0 when the
 * layout does not apply -- more than 32 offsets, an offset without its mirror, more than 16 stored diagonals, or
 * 8 * stored * M > 0.75 * 12 * padded_est bytes.  -1 on bad arguments.  (The device build also requires the values to
 * be exactly symmetric and the columns of every row to ascend.) */
int saena_b200_symdiag_plan(int M, int n_offsets, const int32_t *offsets, int64_t nnz, int64_t padded_est,
                            int32_t *stored);
/* Setup-time choice of every operator's row mapping by measurement: starting from the nnz/row rule, times the
 * neighbouring mappings (1/8 .. 8x the threads per row; the sorted sliced layout where it applies) with `reps`
 * applications each and keeps the fastest where it wins by more than min_gain (e.g. 0.03).  Collective on several
 * ranks (same candidates everywhere, decision on the slowest rank's time, one mapping per operator on all ranks);
 * call after finalize -- and after p2p_import, so that the exchange timed is the one the solve will use.  On one rank
 * it then puts each level on the route (saena_b200_set_level_route) where the three operators stream fewer bytes than
 * the stored one and a Chebyshev sweep through them measures faster by more than min_gain. */
int saena_b200_autotune_mapping(saena_b200_ctx *ctx, int reps, double min_gain, int *changed_out);
/* the mapping in use (same codes) */
int saena_b200_get_mapping(const saena_b200_ctx *ctx, int level, int kind);
/* Level route: level `level`'s operator applied as R_{l-1} (A_{l-1} (P_{l-1} x)), three SpMVs over the operators of the
 * level above, instead of streaming the stored Galerkin product A_l -- fewer bytes where A_l's rows are much longer than
 * the fine level's (level 1 of a 7-point Poisson hierarchy).  Every application of A_l in the solve, the per-operator
 * hooks and the timing loops then take the route, and saena_b200_operator_bytes(level, KIND_A) reports the three
 * operators' bytes; the eigenvalue estimate keeps the stored operator.  One rank, no scaled hierarchy, level >= 1 with
 * no repartition below the level above, no operator with a halo or on the dense path; and R A P must agree with the
 * stored A_l to 1e-12 (relative 2-norm on two seeded random vectors), so that a hierarchy whose A_l is not the product
 * of the operators next to it keeps its own.  saena_b200_autotune_mapping picks the route per level by measurement on
 * one rank; this setter (tests, A/B runs) fails where the conditions or the check do not hold.  finalize resets every
 * level to its stored operator.  get: 1 on the route, 0 not, -1 no such level; ms_stored / ms_route (optional) receive
 * the autotune's median ms of a Chebyshev sweep on the stored operator and on the route (0 where it did not time the
 * level: not eligible, not fewer bytes, or the check failed). */
int saena_b200_set_level_route(saena_b200_ctx *ctx, int level, int on);
int saena_b200_get_level_route(const saena_b200_ctx *ctx, int level, float *ms_stored, float *ms_route);
/* algorithmic bytes of one application of an operator (SURVEY.md 8d formula), for the roofline.  While the
 * preconditioner precision is 32: the FP32 V-cycle's bytes, 4-byte values and vector elements (column ids and row
 * offsets unchanged). */
int64_t saena_b200_operator_bytes(const saena_b200_ctx *ctx, int level, int kind);

/* FP32 preconditioner.  bits = 64 (default) or 32.  At 32, saena_b200_solve_pcg and _pcg_dev apply the preconditioner
 * as an FP32 V-cycle: r is rounded to float, the V-cycle runs from a zero iterate on float vectors and FP32 copies of the
 * operators' values (same smoother, constants, route and graphs; the coarsest level's FP64 solve between two
 * conversions), and its iterate is widened to double.  The Krylov loop stays FP64: the residual recurrence, alpha, beta,
 * the dots, the stop test and u.  solve_vcycle, solve_cg and solve_smoother ignore the switch.  The FP32 copies follow
 * every later update_values, set_mapping, autotune_mapping, set_level_route, set_operator_dense and
 * set_coarsest_solver: they are rebuilt before the next FP32 use.  Refused (non-zero, the switch stays at 64, the
 * reason in last_error): bits other than 32 / 64; several ranks or a detached share; a context not finalized; a scaled
 * hierarchy; a repartitioning level; an operator with a halo, in the merged layout or on streaming row blocks (negative
 * mapping codes); a failed allocation.  finalize resets the switch to 64.  While it is 32 the block solve and its hooks
 * refuse. */
int saena_b200_set_precond_precision(saena_b200_ctx *ctx, int bits);
int saena_b200_get_precond_precision(const saena_b200_ctx *ctx);
/* The per-operator hooks on the FP32 path (float vectors on the host; refused unless the precision is 32):
 * w = Op v, res = A u - rhs, `iters` smoother sweeps on u in place, one FP32 V-cycle on u in place. */
int saena_b200_matvec_f32(saena_b200_ctx *ctx, int level, int kind, const float *v, float *w);
int saena_b200_residual_f32(saena_b200_ctx *ctx, int level, const float *u, const float *rhs, float *res);
int saena_b200_smooth_f32(saena_b200_ctx *ctx, int level, int smoother, int iters, float *u, const float *rhs);
int saena_b200_vcycle_f32(saena_b200_ctx *ctx, int level, int smoother, int pre, int post, float *u, const float *rhs);

#ifdef __cplusplus
}
#endif
#endif
