"""Run under torchrun with N CPU processes (gloo): the row-partitioned setup (saena_b200/sa_setup_dist.py) on N
ranks against the same setup on one rank (sa_setup.build_device_hierarchy, the global hierarchy) on the same matrix.

Every rank builds its share; rank 0 gathers the shares, re-assembles the global operators of every
level from the per-rank reference layout (local block + remote block) and compares them with the
one-rank hierarchy: same level count, same aggregates (identical P patterns), same sparsity patterns,
values to summation order, same Chebyshev bounds.  Then the multi-rank oracle solves on the gathered
shares (halo plan, repartition plan and agglomeration included) and must reproduce the one-rank
oracle's PCG run on the one-rank hierarchy.

With DSC_GPU=1 (one process per GPU, NCCL; tests/test_multigpu.py) the setup runs on the GPUs and every rank
also uploads its share and solves with the CUDA library: same iteration count and residual history as the
multi-rank oracle on the same shares.

usage: dist_setup_check.py poisson <n> | unstructured <g>   [dense|esc] [double]"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from saena_b200 import sa_setup, sa_setup_dist as sd  # noqa: E402


def global_coo(ops):
    """re-assemble (row, col, val) with global ids from every rank's Operator"""
    rows, cols, vals = [], [], []
    for op in ops:
        if op.M == 0:
            continue
        r = np.repeat(np.arange(op.M, dtype=np.int64), op.nnzPerRow_local) + op.row_offset
        rows.append(r); cols.append(op.col_local.astype(np.int64)); vals.append(op.val_local)
        if op.nnz_remote:
            # remote block: column-major; the distinct ghost columns, grouped by owner, are what the owners'
            # vIndex lists name -- recover them from the senders' side
            ghost_cols = []
            for p, cnt in zip(op.recvProcRank, op.recvProcCount):
                peer = ops[int(p)]
                o = int(peer.vdispls[op.rank])
                ghost_cols.append(peer.vIndex[o:o + int(cnt)].astype(np.int64) + peer.col_offset)
                assert int(peer.sendProcCount[list(peer.sendProcRank).index(op.rank)]) == int(cnt)
            ghost_cols = np.concatenate(ghost_cols)
            assert len(ghost_cols) == op.col_remote_size
            rows.append(op.row_remote.astype(np.int64) + op.row_offset)
            cols.append(np.repeat(ghost_cols, op.nnzPerCol_remote)); vals.append(op.val_remote)
    r, c, v = np.concatenate(rows), np.concatenate(cols), np.concatenate(vals)
    order = np.lexsort((c, r))
    return r[order], c[order], v[order]


def main():
    on_gpu = bool(os.environ.get("DSC_GPU"))
    if on_gpu:
        local = int(os.environ.get("LOCAL_RANK", 0))
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        dist.init_process_group("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    what, size = sys.argv[1], int(sys.argv[2])
    dense = True if "dense" in sys.argv[3:] else (False if "esc" in sys.argv[3:] else None)
    float_level = 100 if "double" in sys.argv[3:] else 0
    agg_below = int(os.environ.get("DSC_AGG_BELOW", "150"))
    comm = sd.Comm()
    opts = sa_setup.SetupOptions(float_level=float_level)
    if what == "poisson":
        n, row, col, val = sa_setup.poisson3d_coo(size)
        A0 = sd.poisson3d_dcsr(size, comm)
        rhs = sa_setup.poisson3d_rhs(size)
        # the row generator is the COO generator
        g = sd.coo_dcsr(n, row, col, val, comm)
        assert torch.equal(g.row, A0.row) and torch.equal(g.col, A0.col) and torch.equal(g.val, A0.val)
        assert np.array_equal(sd.poisson3d_rhs_rows(size, A0.r0, A0.r1), rhs[A0.r0:A0.r1])
    else:
        n, row, col, val = sa_setup.unstructured2d_coo(size)
        A0 = sd.coo_dcsr(n, row, col, val, comm)
        rhs = sa_setup.unstructured2d_rhs(n)
    if "skew" in sys.argv[3:]:
        # a lopsided input partition (rank 0 holds 70 % of the rows, one rank none): the setup first moves the
        # matrix to the nnz-balanced partition
        cuts = [0, int(0.7 * n)] + [int(0.7 * n) + (n - int(0.7 * n)) * r // max(world - 2, 1) for r in range(1, world - 1)] + [n]
        cuts = sorted(cuts + [n] * (world + 1 - len(cuts)))[:world + 1]
        cuts[-1] = n
        A0 = sd.coo_dcsr(n, row, col, val, comm, split=np.array(cuts))
    h, summary = sd.build_distributed_hierarchy(A0, opts, agglomerate_below=agg_below, rebalance_above=1.10, dense=dense)
    shares = [None] * world
    dist.gather_object(h, shares if rank == 0 else None, dst=0)
    if rank == 0 and "nocompare" in sys.argv[3:]:
        # sizes the one-rank setup is too slow for on the CPU: the shares must still be a working hierarchy
        from oracle.oracle import Oracle
        on = Oracle(shares)
        parts = [rhs[s.levels[0].A.row_offset:s.levels[0].A.row_offset + s.levels[0].A.M] for s in shares]
        un, itn, hn = on.solve_pcg(parts)
        assert hn[-1] / hn[0] < 1e-8 and itn <= 15, (itn, hn)
        print(f"DIST_SETUP_OK (no comparison) world={world} {what} {size} levels={len(h.levels)} iters={itn} "
              f"rel_res={hn[-1] / hn[0]:.2e}\n" + "\n".join(summary), flush=True)
        expect = [itn, hn]
    elif rank == 0:
        ref = sa_setup.build_device_hierarchy(n, row, col, val, opts, device="cuda" if on_gpu else "cpu")
        assert len(ref.levels) == len(h.levels), (len(ref.levels), len(h.levels))
        for l, lv in enumerate(ref.levels):
            mats = [("A", lv.A, [s.levels[l].A for s in shares])]
            if lv.P is not None:
                mats += [("P", lv.P, [s.levels[l].P for s in shares]), ("R", lv.R, [s.levels[l].R for s in shares])]
            for name, M, ops in mats:
                r, c, v = global_coo(ops)
                assert sum(op.M for op in ops) == M.n_rows and ops[0].Mbig == M.n_rows and ops[0].Nbig == M.n_cols
                rr, cc, vv = M.row.cpu().numpy(), M.col.cpu().numpy(), M.val.cpu().numpy()
                assert len(r) == len(rr), (l, name, len(r), len(rr))
                assert np.array_equal(r, rr) and np.array_equal(c, cc), (l, name, "pattern")
                err = np.max(np.abs(v - vv)) / np.max(np.abs(vv))
                assert err < 1e-13, (l, name, err)
            inv = np.concatenate([s.levels[l].inv_diag for s in shares])
            assert np.allclose(inv, lv.inv_diag.cpu().numpy(), rtol=1e-13, atol=0)
            assert abs(shares[0].levels[l].eig_max - lv.eig_max) < 1e-9 * lv.eig_max, (l, shares[0].levels[l].eig_max, lv.eig_max)
            assert all(s.levels[l].eig_max == shares[0].levels[l].eig_max for s in shares)
            assert all(s.levels[l].A.use_double == lv.a_use_double for s in shares)
        # partition rules: the coarsest on rank 0, levels under the threshold agglomerated, balance kept
        L = len(ref.levels)
        assert shares[0].levels[-1].A.M == ref.levels[-1].A.n_rows
        for l in range(1, L):
            on0 = shares[0].levels[l].A.M == ref.levels[l].A.n_rows
            if ref.levels[l].A.n_rows < agg_below or l == L - 1:
                assert on0, l
        spread = [l for l in range(1, L) if shares[0].levels[l].A.M != ref.levels[l].A.n_rows]
        for l in spread:
            per = np.array([s.levels[l].A.nnz for s in shares], float)
            assert per.max() * world / per.sum() < 1.6, (l, per)
        # the solve: multi-rank oracle on the shares vs one-rank oracle on the one-rank hierarchy
        from oracle.oracle import Oracle
        o1 = Oracle(ref.to_rank(0, 1))
        u1, it1, h1 = o1.solve_pcg(rhs)
        on = Oracle(shares)
        parts = [rhs[s.levels[0].A.row_offset:s.levels[0].A.row_offset + s.levels[0].A.M] for s in shares]
        un, itn, hn = on.solve_pcg(parts)
        assert itn == it1, (itn, it1)
        k = min(len(h1), len(hn))
        # float_level 0: the shares exchange ghost values as float, the one-rank run has no halo at all -- the whole
        # effect of the cast shows (not just a rounding flip); with every halo in double the north_star bound holds
        tol = 1e-9 if float_level else 1e-3
        dev = np.max(np.abs(hn[:k] - h1[:k]) / h1[:k])
        assert dev <= tol, dev
        un = np.concatenate(un)
        assert np.linalg.norm(un - u1) / np.linalg.norm(u1) < 1e-7
        expect = [itn, hn]
    if on_gpu:
        # the CUDA library on the shares the distributed setup produced
        from saena_b200 import native
        from saena_b200.distributed import exchange_nccl_id, setup_p2p_halo
        expect = expect if rank == 0 else [None, None]
        dist.broadcast_object_list(expect, src=0)
        ctx = native.Context(device=local, rank=rank, nranks=world, nccl_id=exchange_nccl_id(native.nccl_unique_id))
        ctx.upload_hierarchy(h)
        setup_p2p_halo(ctx)
        l0 = h.levels[0].A
        u, it_gpu, h_gpu = ctx.solve_pcg(rhs[l0.row_offset:l0.row_offset + l0.M])
        assert it_gpu == expect[0], (it_gpu, expect[0])
        k = min(len(h_gpu), len(expect[1]))
        gdev = np.max(np.abs(np.asarray(h_gpu)[:k] - expect[1][:k]) / expect[1][:k])
        assert gdev <= (1e-9 if float_level else 1e-6), gdev
        dist.barrier()
        ctx.close()
        if rank == 0:
            print(f"DIST_SETUP_GPU_OK hist_dev={gdev:.2e}", flush=True)
    if rank == 0 and "nocompare" not in sys.argv[3:]:
        print(f"DIST_SETUP_OK world={world} {what} {size} levels={L} spread_levels={len(spread) + 1} iters={itn} "
              f"hist_dev={dev:.2e}\n" + "\n".join(summary), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
