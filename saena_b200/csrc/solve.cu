// solve.cu -- smoothers, V-cycle and the Krylov drivers on the uploaded hierarchy.
//
//   saena_object::smooth      /root/reference/include/saena_object.tpp:85-96
//   saena_matrix::chebyshev   /root/reference/src/saena_matrix.cpp:1074-1131
//   saena_matrix::jacobi      /root/reference/src/saena_matrix.cpp:1044-1071
//   saena_object::vcycle      /root/reference/src/saena_object_solve.cpp:961-1431
//   saena_object::solve_pCG   /root/reference/src/saena_object_solve.cpp:2389-2801
//   saena_object::solve       /root/reference/src/saena_object_solve.cpp:1883-2014
//   saena_object::solve_CG    /root/reference/src/saena_object_solve.cpp:2119-2386
//
// Every smoother sweep is ONE pass over A (SpMV with the update fused as epilogue); the iterate
// ping-pongs between two buffers because a fused sweep must read the old u of other rows.  The
// first sweep from a zero iterate (every coarse-level entry and the preconditioner's rho = 0)
// needs no pass over A at all.  Prolongation is fused with the correction u -= P e.
//
// The FP32 preconditioner (saena_b200_set_precond_precision 32) runs the same smoother and V-cycle on float vectors and
// the operators' FP32 copies: sb_apply_level_A, sb_smooth, sb_vcycle and sb_vcycle_from_zero are templates on the value
// type V, instantiated for double and float.  Steps that only exist in FP64 -- repartitions, scaling, the fused residual
// + restriction -- are compiled into the double form only (sb_f32_sync refuses hierarchies that need them), and the
// coarsest level runs its FP64 solve between two conversions.
#include <math.h>

#include <type_traits>

#include "common.h"

// the route's two fine-level intermediates of each precision
static double *route_buf(saena_b200_ctx *ctx, int i, double) { return i ? ctx->route_s : ctx->route_t; }
static float *route_buf(saena_b200_ctx *ctx, int i, float) { return i ? ctx->route32_s : ctx->route32_t; }

// Level l's operator.  Pairwise aggregation halves the rows of the fine level, but the Galerkin product A_l = R A P
// of a short-row operator has far longer rows: on the 256^3 Poisson hierarchy A_1 has 68 entries a row and five times
// A_0's bytes, while P_0, A_0 and R_0 together stream 0.66 of A_1's bytes.  On a route level (DevLevel::route) the product
// is therefore applied as three SpMVs, each operator on its own mapping, through two fine-level intermediates; R's
// rows are level l's rows, so the epilogue (residual, smoother update) fuses into the last one unchanged.  A_{l-1} is
// always the stored operator.
template <typename V>
static int apply_level_A(saena_b200_ctx *ctx, int l, const V *x, int epi, const EpiArgsT<V> &args) {
    DevLevel &lv = ctx->levels[l];
    if (!lv.route) return sb_apply(ctx, lv.A, x, epi, args);
    DevLevel &fl = ctx->levels[l - 1];
    if (ctx->route_cap < fl.M) SB_FAIL("apply: route level without its intermediate vectors");
    V *t = route_buf(ctx, 0, V()), *s = route_buf(ctx, 1, V());
    EpiArgsT<V> e{};
    e.out = t;
    SB_TRY(sb_apply(ctx, fl.P, x, EPI_PLAIN, e));
    e.out = s;
    SB_TRY(sb_apply(ctx, fl.A, t, EPI_PLAIN, e));
    return sb_apply(ctx, fl.R, s, epi, args);
}

int sb_apply_level_A(saena_b200_ctx *ctx, int l, const double *x, int epi, const EpiArgs &args) {
    return apply_level_A(ctx, l, x, epi, args);
}
int sb_apply_level_A(saena_b200_ctx *ctx, int l, const float *x, int epi, const EpiArgs32 &args) {
    return apply_level_A(ctx, l, x, epi, args);
}

int64_t sb_level_A_bytes(const saena_b200_ctx *ctx, int l, int vb) {
    const DevLevel &lv = ctx->levels[l];
    if (!lv.route) return sb_operator_bytes(lv.A, vb);
    const DevLevel &fl = ctx->levels[l - 1];
    return sb_operator_bytes(fl.P, vb) + sb_operator_bytes(fl.A, vb) + sb_operator_bytes(fl.R, vb);
}

template <typename V>
static int smooth(saena_b200_ctx *ctx, int l, int smoother, int iters, const V *rhs, bool u_is_zero) {
    DevLevel &lv = ctx->levels[l];
    if (iters <= 0 || lv.M == 0) {
        if (iters > 0 && (!lv.A.sends.empty() || !lv.A.recvs.empty())) SB_FAIL("smooth: empty rank with a halo plan");
        return 0;
    }
    const LevelVecs<V> v = sb_level_vecs(lv, V());
    EpiArgsT<V> e{};
    e.rhs = rhs;
    e.inv_diag = v.inv_diag;
    if (smoother == SAENA_B200_JACOBI) {
        // u -= (omega D^-1)(A u - rhs), omega = float(2.0/3) promoted (saena_matrix.h:182)
        e.c1 = V((double)(float)(2.0 / 3));
        int j = 0;
        if (u_is_zero) {
            // A*0 = 0: u = 0 - (0 - rhs)*(invd*omega) = (omega*invd)*rhs, no pass over A
            SB_TRY(sb_cheb_first_zero(ctx, lv.M, rhs, v.inv_diag, e.c1, v.d, v.u[lv.cur]));
            j = 1;
        }
        for (; j < iters; ++j) {
            e.u_in = v.u[lv.cur];
            e.out = v.u[lv.cur ^ 1];
            SB_TRY(sb_apply_level_A(ctx, l, v.u[lv.cur], EPI_JACOBI, e));
            lv.cur ^= 1;
        }
        return 0;
    }
    if (smoother != SAENA_B200_CHEBYSHEV) SB_FAIL("smooth: unknown smoother");
    // scalar recurrences exactly as saena_matrix.cpp:1084-1091, :1112-1116
    const double eig = lv.eig_max;
    const double alpha = 0.13 * eig;
    const double beta = eig;
    const double delta = (beta - alpha) / 2.0;
    const double theta = (beta + alpha) / 2.0;
    const double s1 = theta / delta;
    const double twos1 = 2.0 * s1;
    double rhok = 1.0 / s1;
    e.d_in = v.d;
    e.d_out = v.d;
    // first sweep: d = (1/theta) D^-1 (rhs - A u); u += d
    if (u_is_zero) {
        SB_TRY(sb_cheb_first_zero(ctx, lv.M, rhs, v.inv_diag, V(1.0 / theta), v.d, v.u[lv.cur]));
    } else {
        e.c1 = V(1.0 / theta);
        e.u_in = v.u[lv.cur];
        e.out = v.u[lv.cur ^ 1];
        SB_TRY(sb_apply_level_A(ctx, l, v.u[lv.cur], EPI_CHEB_FIRST, e));
        lv.cur ^= 1;
    }
    for (int i = 1; i < iters; ++i) {
        const double rhokp1 = 1.0 / (twos1 - rhok);
        const double two_rhokp1 = 2.0 * rhokp1;
        const double d1 = rhokp1 * rhok;
        const double d2 = two_rhokp1 / delta;
        rhok = rhokp1;
        e.c1 = V(d1);
        e.c2 = V(d2);
        e.u_in = v.u[lv.cur];
        e.out = v.u[lv.cur ^ 1];
        SB_TRY(sb_apply_level_A(ctx, l, v.u[lv.cur], EPI_CHEB_NEXT, e));
        lv.cur ^= 1;
    }
    return 0;
}

int sb_smooth(saena_b200_ctx *ctx, int l, int smoother, int iters, const double *rhs, bool u_is_zero) {
    return smooth(ctx, l, smoother, iters, rhs, u_is_zero);
}
int sb_smooth(saena_b200_ctx *ctx, int l, int smoother, int iters, const float *rhs, bool u_is_zero) {
    return smooth(ctx, l, smoother, iters, rhs, u_is_zero);
}

// V-cycle on grid l with right-hand side `rhs`; the iterate is lv.u[lv.cur] (FP32: lv.u32[lv.cur]) on entry and exit.
template <typename V>
static int vcycle(saena_b200_ctx *ctx, int l, int smoother, int pre, int post, const V *rhs, bool u_is_zero) {
    constexpr bool F64 = std::is_same<V, double>::value;
    const int max_level = (int)ctx->levels.size() - 1;
    DevLevel &lv = ctx->levels[l];
    const LevelVecs<V> v = sb_level_vecs(lv, V());
    // solve.cpp:991-1057 coarsest level: direct solve on the rank that owns it
    if (l == max_level) {
        if constexpr (!F64) {
            // FP32: the FP64 solve between two conversions (res, unused on the coarsest level, holds the FP64 rhs); CG
            // starts from the current iterate
            if (lv.M > 0) {
                SB_TRY(sb_convert(ctx, lv.M, rhs, lv.res));
                if (ctx->coarsest_cg && !u_is_zero) SB_TRY(sb_convert(ctx, lv.M, v.u[lv.cur], lv.u[lv.cur]));
                SB_TRY(sb_vcycle(ctx, l, smoother, pre, post, (const double *)lv.res, u_is_zero));
                SB_TRY(sb_convert(ctx, lv.M, lv.u[lv.cur], v.u[lv.cur]));
            }
            return 0;
        } else {
            SbRange rg(ctx, "coarsest", l);
            if (lv.M > 0 && ctx->coarsest_cg) {
                // direct_solver == "CG" (:998-999): u is the initial guess of solve_coarsest_CG
                if (!lv.A.sends.empty() || !lv.A.recvs.empty()) SB_FAIL("vcycle: the coarsest level must live on one rank");
                if (u_is_zero) SB_TRY(sb_fill_zero(ctx, lv.u[lv.cur], lv.M));
                SB_TRY(sb_coarsest_cg(ctx, rhs, lv.u[lv.cur]));
            } else if (lv.M > 0) {
                if (ctx->coarse_n != lv.M) SB_FAIL("vcycle: no coarsest factor was uploaded for the coarsest level");
                SB_TRY(sb_coarsest_apply(ctx, rhs, lv.u[lv.cur]));
            }
            return 0;
        }
    }
    DevLevel &cl = ctx->levels[l + 1];
    const LevelVecs<V> cv = sb_level_vecs(cl, V());
    // 1. pre-smooth (:1105-1107)
    if (pre) { SbRange rg(ctx, "pre-smooth", l); SB_TRY(sb_smooth(ctx, l, smoother, pre, rhs, u_is_zero)); }
    else if (u_is_zero) SB_TRY(sb_fill_zero(ctx, v.u[lv.cur], lv.M));
    // 2. + 3. residual res = A u - rhs (:1140) and restriction (:1175) into the coarse grid's rhs, through the old
    //    partition if they differ.  Opt-in (saena_b200_set_fused_restrict): both as ONE pass over A that scatters every
    //    fine residual through its row of P and never writes res (fused_restrict.cu; measured in
    //    profiles/r02_fused_restrict.md: -8 % on level 0, +3 % / +37 % on levels 1 / 2 -- off by default, and FP64
    //    atomics make the coarse vector's last bits depend on the run).  Not on a route level: the fused kernel
    //    walks the stored A.
    bool fused_rr = false;
    if constexpr (F64) if (!(pre == 0 && u_is_zero) && ctx->fused_restrict_levels > l && !lv.route) {
        const bool ident = lv.repart.identity();
        const int rc = sb_residual_restrict_fused(ctx, l, lv.u[lv.cur], rhs, ident ? cl.rhs : lv.xfer_old);
        if (rc < 0) SB_FAIL("vcycle: fused residual + restriction failed to launch");
        fused_rr = rc == 1;
        if (fused_rr && !ident) SB_TRY(sb_repart(ctx, lv.repart, false, lv.xfer_old, cl.rhs, ctx->stream));
    }
    // with a zero iterate and no pre-smoothing the residual is -rhs
    if (fused_rr) {
    } else if (pre == 0 && u_is_zero) {
        SB_TRY(sb_negate_copy(ctx, lv.M, rhs, v.res));
    } else {
        SbRange rg(ctx, "residual", l);
        EpiArgsT<V> e{};
        e.rhs = rhs;
        e.out = v.res;
        SB_TRY(sb_apply_level_A(ctx, l, v.u[lv.cur], EPI_RESIDUAL, e));
    }
    if (!fused_rr) {
        SbRange rg(ctx, "Rtransfer", l);
        EpiArgsT<V> e{};
        const bool ident = lv.repart.identity();
        e.out = cv.rhs;
        if constexpr (F64) if (!ident) e.out = lv.xfer_old;
        SB_TRY(sb_apply(ctx, lv.R, v.res, EPI_PLAIN, e));
        if constexpr (F64) if (!ident) SB_TRY(sb_repart(ctx, lv.repart, false, lv.xfer_old, cl.rhs, ctx->stream));  // :1201-1203
    }
    // scale the next level's rhs (:1245-1247)
    if constexpr (F64) if (ctx->scale) SB_TRY(sb_scale_vector(ctx, cl.M, cl.rhs, cl.inv_sq_diag));
    // 4. recurse with a zero initial correction (:1249, :1256)
    SB_TRY(sb_vcycle(ctx, l + 1, smoother, pre, post, (const V *)cv.rhs, true));
    // scale the coarse correction (:1264-1266)
    if constexpr (F64) if (ctx->scale) SB_TRY(sb_scale_vector(ctx, cl.M, cl.u[cl.cur], cl.inv_sq_diag));
    // 5. + 6. prolong and correct: u -= P e_c (:1301-1303, :1325, :1360-1361)
    {
        SbRange rg(ctx, "Ptransfer", l);
        const V *ec = cv.u[cl.cur];
        if constexpr (F64) if (!lv.repart.identity()) {
            SB_TRY(sb_repart(ctx, lv.repart, true, ec, lv.xfer_old, ctx->stream));
            ec = lv.xfer_old;
        }
        EpiArgsT<V> e{};
        e.u_in = v.u[lv.cur];
        e.out = v.u[lv.cur];  // row i reads and writes only u[i]: in place
        SB_TRY(sb_apply(ctx, lv.P, ec, EPI_SUB, e));
    }
    // 7. post-smooth (:1397-1399)
    if (post) { SbRange rg(ctx, "post-smooth", l); SB_TRY(sb_smooth(ctx, l, smoother, post, rhs, false)); }
    return 0;
}

int sb_vcycle(saena_b200_ctx *ctx, int l, int smoother, int pre, int post, const double *rhs, bool u_is_zero) {
    return vcycle(ctx, l, smoother, pre, post, rhs, u_is_zero);
}
int sb_vcycle(saena_b200_ctx *ctx, int l, int smoother, int pre, int post, const float *rhs, bool u_is_zero) {
    return vcycle(ctx, l, smoother, pre, post, rhs, u_is_zero);
}

// Every call that changes what a captured V-cycle would run -- values, layouts, mappings, the route, the coarsest
// solver, Chebyshev bounds -- comes through here, so the FP32 copies are marked stale at the same points
// (sb_f32_sync builds them again before their next use).
void sb_invalidate_graphs(saena_b200_ctx *ctx) {
    for (VcycleGraph &g : ctx->graphs)
        if (g.exec) cudaGraphExecDestroy(g.exec);
    ctx->graphs.clear();
    ctx->f32_stale = true;
}

// Multi-rank capture.  The halo's comm stream is forked from the compute stream by an event at
// every operator application (operator.cu:apply_epi) and so joins the capture; with the
// peer-memory halo nothing joins it back (the hand-over is a flag, p2p_halo.cu), so the capture
// ends with an explicit join.  ncclSend/ncclRecv (Grid::repart_u to the agglomerated levels, or
// the NCCL halo) are captured as NCCL's own graph nodes; every rank captures in the same call.
static int join_comm_stream(saena_b200_ctx *ctx) {
    if (ctx->nranks == 1) return 0;
    cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
    SB_CUDA(cudaStreamIsCapturing(ctx->comm_stream, &st));
    if (st != cudaStreamCaptureStatusActive) return 0;
    SB_CUDA(cudaEventRecord(ctx->ev_halo, ctx->comm_stream));
    SB_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_halo, 0));
    return 0;
}

template <typename V>
static int vcycle_from_zero(saena_b200_ctx *ctx, int smoother, int pre, int post, const V *rhs) {
    const int bits = std::is_same<V, double>::value ? 64 : 32;
    // a zero iterate is overwritten, so every level may start in buffer 0: the launch sequence
    // (pointers included) is then identical from one V-cycle to the next
    for (DevLevel &lv : ctx->levels) lv.cur = 0;
    const bool capturable = ctx->use_graphs && !ctx->coarsest_cg && (ctx->nranks == 1 || ctx->use_graphs_multi);
    if (!capturable) return sb_vcycle(ctx, 0, smoother, pre, post, rhs, true);
    VcycleGraph *known = nullptr;
    for (VcycleGraph &g : ctx->graphs)
        if (g.k == 0 && g.bits == bits && g.rhs == rhs && g.smoother == smoother && g.pre == pre && g.post == post)
            known = &g;
    if (known && known->exec) {
        SB_CUDA(cudaGraphLaunch(known->exec, ctx->stream));
        ctx->launches += known->launches;
        ++ctx->graph_replays;
        for (size_t l = 0; l < ctx->levels.size(); ++l) ctx->levels[l].cur = known->cur_after[l];
        return 0;
    }
    if (!known && ctx->nranks > 1) {
        // several ranks: the first V-cycle of a configuration runs eagerly (NCCL opens its
        // point-to-point channels, every lazy allocation happens), the next one is captured
        ctx->graphs.push_back(VcycleGraph{rhs, smoother, pre, post, nullptr, 0, {}, 0, bits});
        return sb_vcycle(ctx, 0, smoother, pre, post, rhs, true);
    }
    // first use of this configuration (second on several ranks): capture, instantiate, launch
    const int64_t before = ctx->launches;
    cudaGraph_t graph = nullptr;
    SB_CUDA(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
    int rc = sb_vcycle(ctx, 0, smoother, pre, post, rhs, true);
    if (!rc) rc = join_comm_stream(ctx);
    const cudaError_t ce = cudaStreamEndCapture(ctx->stream, &graph);
    auto drop_pending = [&]() {
        for (size_t k = 0; k < ctx->graphs.size(); ++k)
            if (!ctx->graphs[k].exec) { ctx->graphs.erase(ctx->graphs.begin() + k); --k; }
    };
    if (rc || ce != cudaSuccess || !graph) {
        if (graph) cudaGraphDestroy(graph);
        cudaGetLastError();
        ctx->use_graphs = false;  // run eagerly from now on (the capture executed nothing)
        ctx->launches = before;
        drop_pending();
        for (DevLevel &lv : ctx->levels) lv.cur = 0;
        if (rc) return rc;
        ctx->error.clear();
        return sb_vcycle(ctx, 0, smoother, pre, post, rhs, true);
    }
    VcycleGraph g{rhs, smoother, pre, post, nullptr, ctx->launches - before, {}, 0, bits};
    const cudaError_t ie = cudaGraphInstantiate(&g.exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ie != cudaSuccess) {
        cudaGetLastError();
        ctx->use_graphs = false;
        ctx->launches = before;
        drop_pending();
        for (DevLevel &lv : ctx->levels) lv.cur = 0;
        return sb_vcycle(ctx, 0, smoother, pre, post, rhs, true);
    }
    for (DevLevel &lv : ctx->levels) g.cur_after.push_back(lv.cur);
    drop_pending();
    ctx->graphs.push_back(g);
    SB_CUDA(cudaGraphLaunch(g.exec, ctx->stream));
    ++ctx->graph_replays;
    return 0;
}

int sb_vcycle_from_zero(saena_b200_ctx *ctx, int smoother, int pre, int post, const double *rhs) {
    return vcycle_from_zero(ctx, smoother, pre, post, rhs);
}
int sb_vcycle_from_zero(saena_b200_ctx *ctx, int smoother, int pre, int post, const float *rhs) {
    return vcycle_from_zero(ctx, smoother, pre, post, rhs);
}

// ---------------------------------------------------------------------------------------------
// Block forms: k column-major right-hand sides on the levels' block buffers (DevLevel::bu, bd, bres, brhs,
// bxfer_old; column j of a level-l vector at + j * M_l).  Step for step the single code path above -- zero-iterate
// shortcuts, route, repartition, scaling -- with every operator applied once for the k columns (sb_apply_block) and the
// coarsest level solved column by column: column j of every result has the bits of the single path on column j.
// ---------------------------------------------------------------------------------------------
int sb_apply_level_A_block(saena_b200_ctx *ctx, int l, int k, const double *x, int epi, const EpiArgs &args) {
    DevLevel &lv = ctx->levels[l];
    if (!lv.route) return sb_apply_block(ctx, lv.A, k, x, epi, args);
    DevLevel &fl = ctx->levels[l - 1];
    if (ctx->blk_route_cap < (size_t)k * fl.M) SB_FAIL("apply_block: route level without its intermediate vectors");
    EpiArgs e{};
    e.out = ctx->blk_route_t;
    SB_TRY(sb_apply_block(ctx, fl.P, k, x, EPI_PLAIN, e));
    e.out = ctx->blk_route_s;
    SB_TRY(sb_apply_block(ctx, fl.A, k, ctx->blk_route_t, EPI_PLAIN, e));
    return sb_apply_block(ctx, fl.R, k, ctx->blk_route_s, epi, args);
}

int sb_smooth_block(saena_b200_ctx *ctx, int l, int k, int smoother, int iters, const double *rhs, bool u_is_zero) {
    DevLevel &lv = ctx->levels[l];
    if (iters <= 0 || lv.M == 0) return 0;
    EpiArgs e{};
    e.rhs = rhs;
    e.inv_diag = lv.inv_diag;
    if (smoother == SAENA_B200_JACOBI) {
        e.c1 = (double)(float)(2.0 / 3);
        int j = 0;
        if (u_is_zero) {
            SB_TRY(sb_cheb_first_zero_block(ctx, lv.M, k, rhs, lv.inv_diag, e.c1, lv.bd, lv.bu[lv.bcur]));
            j = 1;
        }
        for (; j < iters; ++j) {
            e.u_in = lv.bu[lv.bcur];
            e.out = lv.bu[lv.bcur ^ 1];
            SB_TRY(sb_apply_level_A_block(ctx, l, k, lv.bu[lv.bcur], EPI_JACOBI, e));
            lv.bcur ^= 1;
        }
        return 0;
    }
    if (smoother != SAENA_B200_CHEBYSHEV) SB_FAIL("smooth: unknown smoother");
    const double eig = lv.eig_max;
    const double alpha = 0.13 * eig;
    const double beta = eig;
    const double delta = (beta - alpha) / 2.0;
    const double theta = (beta + alpha) / 2.0;
    const double s1 = theta / delta;
    const double twos1 = 2.0 * s1;
    double rhok = 1.0 / s1;
    e.d_in = lv.bd;
    e.d_out = lv.bd;
    if (u_is_zero) {
        SB_TRY(sb_cheb_first_zero_block(ctx, lv.M, k, rhs, lv.inv_diag, 1.0 / theta, lv.bd, lv.bu[lv.bcur]));
    } else {
        e.c1 = 1.0 / theta;
        e.u_in = lv.bu[lv.bcur];
        e.out = lv.bu[lv.bcur ^ 1];
        SB_TRY(sb_apply_level_A_block(ctx, l, k, lv.bu[lv.bcur], EPI_CHEB_FIRST, e));
        lv.bcur ^= 1;
    }
    for (int i = 1; i < iters; ++i) {
        const double rhokp1 = 1.0 / (twos1 - rhok);
        const double two_rhokp1 = 2.0 * rhokp1;
        const double d1 = rhokp1 * rhok;
        const double d2 = two_rhokp1 / delta;
        rhok = rhokp1;
        e.c1 = d1;
        e.c2 = d2;
        e.u_in = lv.bu[lv.bcur];
        e.out = lv.bu[lv.bcur ^ 1];
        SB_TRY(sb_apply_level_A_block(ctx, l, k, lv.bu[lv.bcur], EPI_CHEB_NEXT, e));
        lv.bcur ^= 1;
    }
    return 0;
}

int sb_vcycle_block(saena_b200_ctx *ctx, int l, int k, int smoother, int pre, int post, const double *rhs,
                    bool u_is_zero) {
    const int max_level = (int)ctx->levels.size() - 1;
    DevLevel &lv = ctx->levels[l];
    const long long M = lv.M;
    if (l == max_level) {
        if (lv.M > 0 && ctx->coarsest_cg) {
            if (u_is_zero) SB_TRY(sb_fill_zero(ctx, lv.bu[lv.bcur], (size_t)k * M));
            for (int j = 0; j < k; ++j) SB_TRY(sb_coarsest_cg(ctx, rhs + j * M, lv.bu[lv.bcur] + j * M));
        } else if (lv.M > 0) {
            if (ctx->coarse_n != lv.M) SB_FAIL("vcycle: no coarsest factor was uploaded for the coarsest level");
            for (int j = 0; j < k; ++j) SB_TRY(sb_coarsest_apply(ctx, rhs + j * M, lv.bu[lv.bcur] + j * M));
        }
        return 0;
    }
    DevLevel &cl = ctx->levels[l + 1];
    const long long Mc = cl.M, Mo = lv.M_coarse_old;
    const bool ident = lv.repart.identity();
    if (pre) SB_TRY(sb_smooth_block(ctx, l, k, smoother, pre, rhs, u_is_zero));
    else if (u_is_zero) SB_TRY(sb_fill_zero(ctx, lv.bu[lv.bcur], (size_t)k * M));
    if (pre == 0 && u_is_zero) {
        SB_TRY(sb_negate_copy_block(ctx, lv.M, k, rhs, lv.bres));
    } else {
        EpiArgs e{};
        e.rhs = rhs;
        e.out = lv.bres;
        SB_TRY(sb_apply_level_A_block(ctx, l, k, lv.bu[lv.bcur], EPI_RESIDUAL, e));
    }
    {
        EpiArgs e{};
        e.out = ident ? cl.brhs : lv.bxfer_old;
        SB_TRY(sb_apply_block(ctx, lv.R, k, lv.bres, EPI_PLAIN, e));
        if (!ident)
            for (int j = 0; j < k; ++j)
                SB_TRY(sb_repart(ctx, lv.repart, false, lv.bxfer_old + j * Mo, cl.brhs + j * Mc, ctx->stream));
    }
    if (ctx->scale) SB_TRY(sb_scale_vector_block(ctx, cl.M, k, cl.brhs, cl.inv_sq_diag));
    SB_TRY(sb_vcycle_block(ctx, l + 1, k, smoother, pre, post, cl.brhs, true));
    if (ctx->scale) SB_TRY(sb_scale_vector_block(ctx, cl.M, k, cl.bu[cl.bcur], cl.inv_sq_diag));
    {
        const double *ec = cl.bu[cl.bcur];
        if (!ident) {
            for (int j = 0; j < k; ++j)
                SB_TRY(sb_repart(ctx, lv.repart, true, ec + j * Mc, lv.bxfer_old + j * Mo, ctx->stream));
            ec = lv.bxfer_old;
        }
        EpiArgs e{};
        e.u_in = lv.bu[lv.bcur];
        e.out = lv.bu[lv.bcur];
        SB_TRY(sb_apply_block(ctx, lv.P, k, ec, EPI_SUB, e));
    }
    if (post) SB_TRY(sb_smooth_block(ctx, l, k, smoother, post, rhs, false));
    return 0;
}

// One rank only (the block calls refuse several), so the first use of a configuration is captured at once.  The key
// is (rhs, smoother, pre, post, k): the block buffers a graph points into stay put until they grow, and growing them
// drops every block graph (sb_block_reserve).
int sb_vcycle_block_from_zero(saena_b200_ctx *ctx, int k, int smoother, int pre, int post, const double *rhs) {
    for (DevLevel &lv : ctx->levels) lv.bcur = 0;
    if (!ctx->use_graphs || ctx->coarsest_cg) return sb_vcycle_block(ctx, 0, k, smoother, pre, post, rhs, true);
    for (VcycleGraph &g : ctx->graphs)
        if (g.k == k && g.rhs == rhs && g.smoother == smoother && g.pre == pre && g.post == post) {
            SB_CUDA(cudaGraphLaunch(g.exec, ctx->stream));
            ctx->launches += g.launches;
            ++ctx->graph_replays;
            for (size_t l = 0; l < ctx->levels.size(); ++l) ctx->levels[l].bcur = g.cur_after[l];
            return 0;
        }
    const int64_t before = ctx->launches;
    cudaGraph_t graph = nullptr;
    SB_CUDA(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
    const int rc = sb_vcycle_block(ctx, 0, k, smoother, pre, post, rhs, true);
    const cudaError_t ce = cudaStreamEndCapture(ctx->stream, &graph);
    cudaGraphExec_t exec = nullptr;
    const cudaError_t ie = (rc || ce != cudaSuccess || !graph) ? cudaErrorUnknown : cudaGraphInstantiate(&exec, graph, 0);
    if (graph) cudaGraphDestroy(graph);
    if (ie != cudaSuccess) {
        // the capture executed nothing: run eagerly (a failed capture of the block V-cycle leaves the single one's
        // graphs as they are)
        cudaGetLastError();
        ctx->launches = before;
        for (DevLevel &lv : ctx->levels) lv.bcur = 0;
        if (rc) return rc;
        ctx->error.clear();
        return sb_vcycle_block(ctx, 0, k, smoother, pre, post, rhs, true);
    }
    VcycleGraph g{rhs, smoother, pre, post, exec, ctx->launches - before, {}, k};
    for (DevLevel &lv : ctx->levels) g.cur_after.push_back(lv.bcur);
    ctx->graphs.push_back(g);
    SB_CUDA(cudaGraphLaunch(g.exec, ctx->stream));
    ++ctx->graph_replays;
    return 0;
}
