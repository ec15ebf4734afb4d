"""The smoothed-aggregation setup of sa_setup.py (whose header cites the reference lines), row-partitioned, one
process per GPU -- ONLY to feed the benchmark, among others with a hierarchy no single GPU can build
(BASELINE.json configs[2]: 512^3 unknowns on 8 B200).  This is the only copy of the setup's steps and level loop:
sa_setup.build_device_hierarchy runs them on one rank (a one-rank `Comm` even inside a process group), where the
collectives are identities, `ColMap` has no ghosts and the aggregation refreshes no ghost states.

The AMG setup is outside this package's scope (see sa_setup.py's header); this module is plumbing made of
torch tensor ops and torch.distributed collectives (NCCL on GPUs, gloo in the CPU tests).  Nothing in the
solve path imports it.

Every step works on a 1-D row partition, with the reference's rules and the same synchronous iterations on any
number of ranks:

  * strength of connection, prolongator, filter: row-local, the values a row needs from other
    ranks (its neighbours' row maxima, aggregate ids, inverse diagonal) are fetched once;
  * aggregation: aggregation_1_dist (src/saena_object_setup1.cpp:724-995) IS a synchronous
    data-parallel iteration -- each round reads the states of the round before -- so exchanging
    the states of the ghost nodes after every round reproduces the one-rank aggregates exactly,
    whatever the partition (tests/dist_setup_check.py compares N ranks with one);
  * coarse numbering: a root's coarse id is its rank among the sorted roots, so each rank's
    aggregates are a contiguous block of coarse rows -- "an aggregate lives where its root lives",
    splitNew in aggregate_index_update (src/saena_object_setup1.cpp:2124-2132);
  * Galerkin product: rows of P for the ghost columns of A are fetched, A P is row-local, and
    R (A P) is formed as P_local^T (A P)_local with the partial coarse rows sent to their owners
    and added there (the reference's distributed matmat moves blocks of B around a ring instead,
    src/saena_object_setup_matmat.cpp:27-1160; the sum is the same up to its order);
  * Chebyshev bound: Lanczos on D^-1/2 A D^-1/2 from the same seeded global start vector.

The partition each level ends up with is the one the solve uses (hierarchy.partition_hierarchy's
rules, hierarchy.coarse_placement): level 0 nnz-balanced, a coarse level follows the level above unless
one rank would hold more than `rebalance_above` x the mean nnz (then it is re-split by its own nnz
balance and moved), levels below `agglomerate_below` global rows and the coarsest live on rank 0.
`coarsen` is the level loop and hands out each level's tensors; `build_distributed_hierarchy` turns
them into each rank's `Hierarchy` in the reference layout, ready for `saena_b200_upload_operator`.
"""
from __future__ import annotations

import os
import sys
import time
from typing import List, Optional, Sequence

import numpy as np
import torch
import torch.distributed as dist

from .hierarchy import F64, I64, KIND_A, KIND_P, KIND_R, Hierarchy, Level, Operator, coarse_placement, repart_plan
from .sa_setup import (ALMOST_ZERO, BIG, JACOBI_OMEGA, DeviceLevel, SetupOptions, _coalesce, _Csr, _expand_segments,
                       _native_spgemm_enabled, _spgemm, _to_torch_csr, _transpose, rank_layout)


# ------------------------------------------------------------------------------------------
# collectives
# ------------------------------------------------------------------------------------------
class Comm:
    """the few collectives the setup needs, on whatever backend the default group runs; `one_rank`: this process
    alone (world size 1) even where a process group runs -- the setup of sa_setup.build_device_hierarchy"""

    def __init__(self, device: Optional[torch.device] = None, one_rank: bool = False):
        self.on = not one_rank and dist.is_available() and dist.is_initialized()
        self.rank = dist.get_rank() if self.on else 0
        self.world = dist.get_world_size() if self.on else 1
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device()) if (self.on and dist.get_backend() == "nccl") \
                else torch.device("cpu")
        self.dev = device

    def all_to_all_counts(self, counts: Sequence[int]) -> List[int]:
        if self.world == 1:
            return list(counts)
        s = torch.tensor(list(counts), dtype=torch.int64, device=self.dev)
        r = torch.empty_like(s)
        dist.all_to_all_single(r, s)
        return [int(x) for x in r.tolist()]

    def all_to_all(self, send: torch.Tensor, send_counts: Sequence[int], recv_counts: Sequence[int]) -> torch.Tensor:
        """send is the concatenation of the pieces for rank 0, 1, ...; returns the concatenation of what they sent"""
        if self.world == 1:
            return send
        out = torch.empty(int(sum(recv_counts)), dtype=send.dtype, device=send.device)
        dist.all_to_all_single(out, send.contiguous(), [int(c) for c in recv_counts], [int(c) for c in send_counts])
        return out

    def sum(self, x):
        """sum of a python number over ranks"""
        if self.world == 1:
            return x
        isint = isinstance(x, (int, np.integer))
        t = torch.tensor([x], dtype=torch.int64 if isint else torch.float64, device=self.dev)
        dist.all_reduce(t)
        return int(t.item()) if isint else float(t.item())

    def norm(self, x: torch.Tensor) -> float:
        """2-norm of a row-partitioned vector"""
        if self.world == 1:
            return float(torch.linalg.norm(x))
        return float(np.sqrt(self.sum(float(torch.dot(x, x)))))

    def sum_tensor(self, t: torch.Tensor) -> torch.Tensor:
        if self.world > 1:
            dist.all_reduce(t)
        return t

    def gather_ints(self, x: int) -> np.ndarray:
        if self.world == 1:
            return np.array([x], I64)
        t = torch.tensor([int(x)], dtype=torch.int64, device=self.dev)
        out = torch.empty(self.world, dtype=torch.int64, device=self.dev)
        dist.all_gather_into_tensor(out, t)
        return out.cpu().numpy().astype(I64)

    def bcast_float(self, x: float, src: int = 0) -> float:
        if self.world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=self.dev)
        dist.broadcast(t, src)
        return float(t.item())

    def bcast_tensor(self, t: Optional[torch.Tensor], dtype, src: int = 0) -> torch.Tensor:
        if self.world == 1:
            return t
        n = torch.tensor([t.numel() if self.rank == src else 0], dtype=torch.int64, device=self.dev)
        dist.broadcast(n, src)
        buf = t.to(self.dev, dtype).contiguous() if self.rank == src else torch.empty(int(n.item()), dtype=dtype, device=self.dev)
        dist.broadcast(buf, src)
        return buf


def _owner(split_t: torch.Tensor, ids: torch.Tensor) -> torch.Tensor:
    """rank owning each global id under a split with possibly empty blocks"""
    return torch.searchsorted(split_t, ids, right=True) - 1


class Fetcher:
    """values of a row-partitioned vector at a fixed list of global ids (sorted ascending): the list is
    sent to the owners once, every fetch is then one all-to-all"""

    def __init__(self, comm: Comm, split: np.ndarray, ids: torch.Tensor):
        self.comm = comm
        split_t = torch.as_tensor(np.asarray(split, I64), device=ids.device)
        own = _owner(split_t, ids)
        self.req_counts = [int(c) for c in torch.bincount(own, minlength=comm.world).tolist()] if ids.numel() else [0] * comm.world
        self.serve_counts = comm.all_to_all_counts(self.req_counts)
        asked = comm.all_to_all(ids, self.req_counts, self.serve_counts)
        self.serve_idx = asked - int(split[comm.rank])          # local ids, grouped by the asking rank

    def fetch(self, x_local: torch.Tensor) -> torch.Tensor:
        return self.comm.all_to_all(x_local[self.serve_idx], self.serve_counts, self.req_counts)


class ColMap:
    """The columns a rank's rows touch, as one index space ordered like the global ids:
    [ghosts below my block | my block | ghosts above].  Monotone in the global id, so row-major
    sorted entries stay sorted and `smallest neighbour` means the same thing in both numberings."""

    def __init__(self, comm: Comm, split: np.ndarray, cols: torch.Tensor):
        self.c0, self.c1 = int(split[comm.rank]), int(split[comm.rank + 1])
        self.m = self.c1 - self.c0
        out = cols[(cols < self.c0) | (cols >= self.c1)]
        self.ghost = torch.unique(out)                                   # sorted
        self.g_lo = int((self.ghost < self.c0).sum()) if self.ghost.numel() else 0
        self.n_ext = self.m + int(self.ghost.numel())
        self.fetcher = Fetcher(comm, split, self.ghost)

    def to_ext(self, gid: torch.Tensor) -> torch.Tensor:
        if not self.ghost.numel():          # every column is mine (one rank): no copy of the column ids at c0 = 0
            return gid - self.c0 if self.c0 else gid
        pos = torch.searchsorted(self.ghost, gid)
        own = (gid >= self.c0) & (gid < self.c1)
        return torch.where(own, gid - self.c0 + self.g_lo, torch.where(gid < self.c0, pos, pos + self.m))

    def extend(self, x_local: torch.Tensor) -> torch.Tensor:
        g = self.fetcher.fetch(x_local)
        return torch.cat([g[:self.g_lo], x_local, g[self.g_lo:]])

    def ghost_ext_index(self) -> torch.Tensor:
        k = torch.arange(self.ghost.numel(), device=self.ghost.device)
        return torch.where(k < self.g_lo, k, k + self.m)


class DCsr:
    """this rank's rows of a row-partitioned matrix: LOCAL row ids, GLOBAL column ids, sorted row-major"""

    def __init__(self, n_rows, n_cols, split, rank, row, col, val):
        self.n_rows, self.n_cols, self.split, self.rank = n_rows, n_cols, np.asarray(split, I64), rank
        self.r0, self.r1 = int(self.split[rank]), int(self.split[rank + 1])
        self.m = self.r1 - self.r0
        self.row, self.col, self.val = row, col, val

    @property
    def nnz(self):
        return int(self.val.numel())

    def counts(self):
        return torch.bincount(self.row, minlength=self.m)

    def ptr(self):
        p = torch.zeros(self.m + 1, dtype=torch.int64, device=self.val.device)
        p[1:] = torch.cumsum(self.counts(), 0)
        return p


def _route_rows(comm: Comm, split_new: np.ndarray, grow: torch.Tensor, *payload: torch.Tensor):
    """send entries to the owner of their GLOBAL row under split_new; returns (grow, *payload) received,
    concatenated in source-rank order"""
    dev = grow.device
    st = torch.as_tensor(np.asarray(split_new, I64), device=dev)
    own = _owner(st, grow)
    if grow.numel() > 1 and not bool((own[1:] >= own[:-1]).all()):
        order = torch.argsort(own, stable=True)
        own, grow = own[order], grow[order]
        payload = tuple(p[order] for p in payload)
    sc = [int(c) for c in torch.bincount(own, minlength=comm.world).tolist()] if grow.numel() else [0] * comm.world
    rc = comm.all_to_all_counts(sc)
    return (comm.all_to_all(grow, sc, rc),) + tuple(comm.all_to_all(p, sc, rc) for p in payload)


def repartition(comm: Comm, A: DCsr, split_new: np.ndarray) -> DCsr:
    """move the rows of A to another row partition (what saena_matrix::repart does to Ac,
    src/saena_matrix_repart.cpp:728-979)"""
    split_new = np.asarray(split_new, I64)
    if np.array_equal(split_new, A.split):
        return A
    grow, col, val = _route_rows(comm, split_new, A.row + A.r0, A.col, A.val)   # sources are ordered: stays sorted
    return DCsr(A.n_rows, A.n_cols, split_new, A.rank, grow - int(split_new[A.rank]), col, val)


def balanced_split_dist(comm: Comm, A: DCsr) -> np.ndarray:
    """hierarchy.balanced_split on a distributed matrix: cut where the running nnz count crosses r/nprocs"""
    nprocs = comm.world
    local = A.nnz
    per = comm.gather_ints(local)
    total, before = int(per.sum()), int(per[:comm.rank].sum())
    cum = torch.cumsum(A.counts(), 0) + before                         # indptr[1:] of my rows, global
    targets = torch.as_tensor(np.arange(1, nprocs, dtype=np.float64) * total / nprocs, device=cum.device)
    below = torch.searchsorted(cum.to(torch.float64), targets, right=False)   # my rows with cum < target
    below = comm.sum_tensor(below.to(torch.int64)).cpu().numpy()
    cuts = np.minimum(below + 1, A.n_rows)
    split = np.concatenate(([0], cuts, [A.n_rows])).astype(I64)
    return np.maximum.accumulate(split)


def fetch_rows(comm: Comm, P: DCsr, cm: ColMap) -> _Csr:
    """rows of P for every index of cm's extended space (my own rows in the middle, the ghost rows fetched
    from their owners), as a matrix with n_ext rows"""
    if comm.world == 1:
        return _Csr(P.m, P.n_cols, P.row, P.col, P.val)
    dev = P.val.device
    f = cm.fetcher
    counts = P.counts()
    ptr = torch.zeros(P.m + 1, dtype=torch.int64, device=dev)
    ptr[1:] = torch.cumsum(counts, 0)
    g_counts = f.fetch(counts)                                           # entries of each ghost row
    e, _ = _expand_segments(ptr, f.serve_idx)
    # entries per asking rank
    served_rows_cum = np.concatenate(([0], np.cumsum(f.serve_counts)))
    cnt_served = counts[f.serve_idx]
    ccum = torch.zeros(f.serve_idx.numel() + 1, dtype=torch.int64, device=dev)
    ccum[1:] = torch.cumsum(cnt_served, 0)
    bounds = ccum[torch.as_tensor(served_rows_cum, device=dev)].tolist()
    sc = [int(bounds[i + 1] - bounds[i]) for i in range(comm.world)]
    rc = comm.all_to_all_counts(sc)
    gcol = comm.all_to_all(P.col[e], sc, rc)
    gval = comm.all_to_all(P.val[e], sc, rc)
    grow = torch.repeat_interleave(cm.ghost_ext_index(), g_counts, output_size=int(gcol.numel()))
    n_lo = int(g_counts[:cm.g_lo].sum()) if cm.g_lo else 0
    row = torch.cat([grow[:n_lo], P.row + cm.g_lo, grow[n_lo:]])
    col = torch.cat([gcol[:n_lo], P.col, gcol[n_lo:]])
    val = torch.cat([gval[:n_lo], P.val, gval[n_lo:]])
    return _Csr(cm.n_ext, P.n_cols, row, col, val)


# ------------------------------------------------------------------------------------------
# the setup steps, row-partitioned
# ------------------------------------------------------------------------------------------
def diag_local(A: DCsr) -> torch.Tensor:
    d = torch.zeros(A.m, dtype=torch.float64, device=A.val.device)
    on = (A.row + A.r0) == A.col
    d[A.row[on]] = A.val[on]
    return d


def lanczos_eig_max_dist(comm: Comm, A: DCsr, cm: ColMap, col_ext: torch.Tensor, inv_diag: torch.Tensor, iters: int,
                         seed: int) -> float:
    """largest eigenvalue of D^-1/2 A D^-1/2 (find_eig: scale_matrix + find_eig_lamlan), x 1.0001; the start vector is
    the same global seeded vector on any number of ranks"""
    dev = A.val.device
    n = A.n_rows
    s = torch.sqrt(inv_diag.abs())
    g = torch.Generator(device="cpu").manual_seed(seed)
    v = torch.randn(n, dtype=torch.float64, generator=g)[A.r0:A.r1].to(dev)
    v = v / comm.norm(v)
    v_prev = torch.zeros_like(v)
    alphas, betas = [], []
    beta = 0.0
    for _ in range(min(iters, n)):
        x = cm.extend(s * v)
        w = torch.zeros(A.m, dtype=torch.float64, device=dev)
        w.index_add_(0, A.row, A.val * x[col_ext])
        w = s * w - beta * v_prev
        alpha = comm.sum(float(torch.dot(w, v)))
        w = w - alpha * v
        beta = comm.norm(w)
        alphas.append(alpha)
        if beta < 1e-14:
            break
        betas.append(beta)
        v_prev, v = v, w / beta
    k = len(alphas)
    T = np.diag(alphas) + np.diag(betas[:k - 1], 1) + np.diag(betas[:k - 1], -1)
    return comm.bcast_float(1.0001 * float(np.linalg.eigvalsh(T)[-1]))


def strength_graph_dist(A: DCsr, cm: ColMap, col_ext: torch.Tensor, conn_str: float):
    """strong off-diagonal connections (row, col) -- create_strength_matrix + setup_matrix -- in cm's extended
    numbering"""
    dev = A.val.device
    off = (A.row + A.r0) != A.col
    max_per_row = torch.full((A.m,), -torch.finfo(torch.float64).max, dtype=torch.float64, device=dev)
    max_per_row.scatter_reduce_(0, A.row[off], -A.val[off], reduce="amax")
    mpr_ext = cm.extend(max_per_row)
    s_row = -A.val / max_per_row[A.row]      # entry   (normalised by its row's maximum)
    s_col = -A.val / mpr_ext[col_ext]        # entryT  (normalised by the column index's row maximum)
    strong = off & ((s_row > conn_str) | (s_col > conn_str))
    return A.row[strong] + cm.g_lo, col_ext[strong]


def aggregate_dist(comm: Comm, cm: ColMap, s_row: torch.Tensor, s_col: torch.Tensor):
    """aggregation_1_dist.  The reference sweeps every undecided node in every round; a node's outcome can only change
    when one of its neighbours was decided in the round before, so only those nodes are re-evaluated here (same rule,
    same synchronous updates, hence the same aggregates -- tests/test_sa_setup.py compares with the reference's).  On
    several ranks the states of the ghost nodes are refreshed after every round.  Returns (coarse id of every node of
    the extended space, number of aggregates, coarse split, rounds)."""
    dev = s_row.device
    E, m, lo = cm.n_ext, cm.m, cm.g_lo
    # CSR of the strength graph by row (s_row is ascending: A is row-major sorted) and by column
    ptr = torch.zeros(E + 1, dtype=torch.int64, device=dev)
    ptr[1:] = torch.cumsum(torch.bincount(s_row, minlength=E), 0)
    order = torch.argsort(s_col, stable=True)
    t_nb = s_row[order]                      # rows that list node j as a neighbour, grouped by j
    tptr = torch.zeros(E + 1, dtype=torch.int64, device=dev)
    tptr[1:] = torch.cumsum(torch.bincount(s_col, minlength=E), 0)
    del order
    agg = torch.arange(E, dtype=torch.int64, device=dev)
    decided = torch.zeros(E, dtype=torch.bool, device=dev)
    is_root = torch.zeros(E, dtype=torch.bool, device=dev)
    ghost_idx = cm.ghost_ext_index()
    F = torch.arange(lo, lo + m, dtype=torch.int64, device=dev)   # undecided nodes to evaluate this round
    rounds = 0
    while comm.sum(int(F.numel())) > 0:
        rounds += 1
        e, seg = _expand_segments(ptr, F)
        nb = s_col[e]
        # eligible neighbours: undecided or root; their aggregate value is their own index
        elig = (~decided[nb]) | is_root[nb]
        cand = torch.where(elig, nb, torch.full_like(nb, BIG))
        mn = torch.full((F.numel(),), BIG, dtype=torch.int64, device=dev)
        mn.scatter_reduce_(0, seg, cand, reduce="amin")
        take = mn < F                                    # a smaller eligible neighbour exists
        mc = torch.where(take, mn, F)
        dec_nei = torch.where(take, decided[mc], torch.ones_like(take))
        root_nei = take & is_root[mc]
        new_root = dec_nei & (~take)
        join = dec_nei & root_nei
        newly = F[dec_nei]
        # synchronous update: everything above read the state of the previous round
        agg[F[join]] = mc[join]
        is_root[F[new_root]] = True
        decided[newly] = True
        # the other ranks' nodes I read: their state after this round
        if comm.world > 1:
            state = decided[lo:lo + m].to(torch.int64) + 2 * is_root[lo:lo + m].to(torch.int64)
            g = cm.fetcher.fetch(state)
            g_dec = (g & 1).bool()
            changed = ghost_idx[g_dec & ~decided[ghost_idx]]
            decided[ghost_idx] = g_dec
            is_root[ghost_idx] = (g & 2).bool()
            newly = torch.cat([newly, changed])
        # next round: undecided nodes one of whose neighbours was just decided
        te, _ = _expand_segments(tptr, newly)
        cand_rows = t_nb[te]
        cand_rows = cand_rows[~decided[cand_rows]]
        F = torch.unique(cand_rows)
    assert bool(decided[lo:lo + m].all())
    # aggregate_index_update: coarse id = rank of the root among the sorted roots (my roots are a block)
    roots_own = is_root[lo:lo + m]
    per = comm.gather_ints(int(roots_own.sum()))
    coarse_split = np.concatenate(([0], np.cumsum(per))).astype(I64)
    coarse_of_own = torch.cumsum(roots_own.to(torch.int64), 0) - 1 + int(coarse_split[comm.rank])
    coarse_of_ext = cm.extend(coarse_of_own)                  # valid at roots, mine and the ghosts'
    agg_c_own = coarse_of_ext[agg[lo:lo + m]]
    return cm.extend(agg_c_own), int(coarse_split[-1]), coarse_split, rounds


def prolongator_dist(A: DCsr, col_ext: torch.Tensor, agg_c_ext: torch.Tensor, nc: int, inv_diag: torch.Tensor) -> DCsr:
    """SA(): P = (I - w D^-1 A) P_t with P_t(i, agg(i)) = 1, on my rows"""
    v = -JACOBI_OMEGA * inv_diag[A.row] * A.val
    v = torch.where((A.row + A.r0) == A.col, v + 1.0, v)
    P = _coalesce(max(A.m, 1), nc, A.row, agg_c_ext[col_ext], v)
    keep = P.val.abs() > ALMOST_ZERO
    return DCsr(A.n_rows, nc, A.split, A.rank, P.row[keep], P.col[keep], P.val[keep])


def transpose_dist(comm: Comm, P: DCsr, coarse_split: np.ndarray) -> DCsr:
    """R = P^T, its rows (coarse) partitioned by coarse_split"""
    grow, gcol, val = _route_rows(comm, coarse_split, P.col, P.row + P.r0, P.val)
    c0 = int(coarse_split[comm.rank])
    key = (grow - c0) * P.n_rows + gcol
    key, order = torch.sort(key)
    return DCsr(P.n_cols, P.n_rows, coarse_split, comm.rank, key // P.n_rows, key % P.n_rows, val[order])


def _add_partial_rows(comm: Comm, nc: int, coarse_split: np.ndarray, grow, gcol, val) -> DCsr:
    """partial coarse rows (global ids) -> their owners, duplicates added"""
    if comm.world == 1:                  # whole rows, already sorted and without duplicates
        return DCsr(nc, nc, coarse_split, 0, grow, gcol, val)
    grow, gcol, val = _route_rows(comm, coarse_split, grow, gcol, val)
    c0 = int(coarse_split[comm.rank])
    mc = int(coarse_split[comm.rank + 1]) - c0
    C = _coalesce(max(mc, 1), nc, grow - c0, gcol, val)
    return DCsr(nc, nc, coarse_split, comm.rank, C.row, C.col, C.val)


# measured on one B200 at 256^3: level 3 -> 4 through sparse x dense products,
# 167 M stored entries x 21 466 columns in 2.5 s ~ 1.4e12 multiply-adds/s; the expand / sort / compress route
# does a few 1e9 scalar products per second (level 2 -> 3: 7.4 s)
_SPMM_FMA_PER_S = 1.4e12
_ESC_PRODUCTS_PER_S = 5e9


def _prefer_dense(comm: Comm, A: DCsr, A_x: _Csr, P: DCsr, P_ext: _Csr, nc: int) -> bool:
    """Which of the two tensor-op routes of galerkin_dist is cheaper for the slowest rank.  On the CPU: expand / sort /
    compress on one rank (the hierarchies the goldens and the CPU suite compare against), and on several ranks
    sparse x dense on small nearly dense levels, so that the gloo tests exercise both routes."""
    dev = A.val.device
    if dev.type != "cuda":
        if comm.world == 1:
            return False
        a_nnz, p_nnz = comm.sum(A.nnz), comm.sum(P.nnz)
        return (a_nnz / max(A.n_rows, 1)) * (p_nnz / max(P.n_rows, 1)) > 4 * nc and A.n_rows <= 20000
    prod_ap = int(P_ext.counts()[A_x.col].sum()) if A.nnz else 0          # scalar products of A P on my rows
    t = torch.tensor([float(prod_ap), float(A.nnz + P.nnz)], dtype=torch.float64, device=dev)
    if comm.world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    prod_ap, nnz_ap = t.tolist()
    # P^T (A P) costs a multiple of A P on these hierarchies (rows of A P are longer than rows of P)
    est_esc = 4.0 * prod_ap / _ESC_PRODUCTS_PER_S
    est_dense = nnz_ap * nc / _SPMM_FMA_PER_S + (8.0 * nc * nc / 2e11 if comm.world > 1 else 0.0)
    return est_dense < est_esc


def galerkin_dist(comm: Comm, A: DCsr, cm: ColMap, col_ext: torch.Tensor, P: DCsr, coarse_split: np.ndarray,
                  dense: Optional[bool] = None, dense_budget_bytes: float = 24e9, verbose: bool = False) -> DCsr:
    """Ac = P^T A P.  On the deep levels of a 3D hierarchy the product is nearly dense (256^3 Poisson, level 3 -> 4:
    rows of A P have ~20 000 entries, 8e11 scalar products) and the sparse expansion drowns; there the products are
    done as sparse x dense, column block by column block, and the result is re-sparsified (structural zeros stay
    exact zeros, so the pattern is the sparse product's barring exact cancellation).  `dense` None: the library's
    device SpGEMM where _native_spgemm_enabled, else _prefer_dense decides."""
    dev = A.val.device
    nc = P.n_cols
    # tests shrink both work sizes so that several column blocks / product chunks are exercised on small inputs
    dense_budget_bytes = float(os.environ.get("SAENA_SETUP_DENSE_BUDGET", dense_budget_bytes))
    chunk = int(os.environ.get("SAENA_SETUP_CHUNK_PRODUCTS", 300_000_000))
    P_ext = fetch_rows(comm, P, cm)
    A_x = _Csr(A.m, cm.n_ext, A.row, col_ext, A.val)
    native = _native_spgemm_enabled(dev, comm.world)
    if dense is None:
        dense = not native and _prefer_dense(comm, A, A_x, P, P_ext, nc)
    uc, inv = torch.unique(P.col, return_inverse=True)                 # coarse rows my P rows reach
    Pt = _transpose(_Csr(A.m, max(int(uc.numel()), 1), P.row, inv, P.val))        # compact coarse rows x my fine rows
    del inv
    if not dense:
        AP = _spgemm(A_x, P_ext, chunk, native)
        C = _spgemm(Pt, AP, chunk, native)
        del AP
        return _add_partial_rows(comm, nc, coarse_split, uc[C.row] if C.nnz else C.row, C.col, C.val)
    # dense column blocks: AP[:, c0:c1] = A_x P_ext[:, c0:c1]; partial coarse rows P_local^T AP summed over ranks
    # the block width must be the same on every rank (one all-reduce per block): sized for the largest rank
    rows_here = torch.tensor([cm.n_ext + A.m], dtype=torch.int64, device=dev)
    if comm.world > 1:
        dist.all_reduce(rows_here, op=dist.ReduceOp.MAX)
    w = int(max(1, min(nc, dense_budget_bytes / 8 / max(int(rows_here.item()) + nc, 1))))
    A_csr = _to_torch_csr(A_x) if A.m else None
    Pt_csr = _to_torch_csr(_transpose(_Csr(A.m, nc, P.row, P.col, P.val))) if A.m else None
    c0r, c1r = int(coarse_split[comm.rank]), int(coarse_split[comm.rank + 1])
    rows, cols, vals = [], [], []
    for b0 in range(0, nc, w):
        b1 = min(nc, b0 + w)
        sel = (P_ext.col >= b0) & (P_ext.col < b1)
        Pd = torch.zeros(cm.n_ext, b1 - b0, dtype=torch.float64, device=dev)
        Pd[P_ext.row[sel], P_ext.col[sel] - b0] = P_ext.val[sel]
        if A.m:
            AP = torch.sparse.mm(A_csr, Pd)
            del Pd
            Cb = torch.sparse.mm(Pt_csr, AP)
            del AP
        else:
            del Pd
            Cb = torch.zeros(nc, b1 - b0, dtype=torch.float64, device=dev)
        comm.sum_tensor(Cb)
        mine = Cb[c0r:c1r]
        idx = torch.nonzero(mine, as_tuple=True)
        rows.append(idx[0]); cols.append(idx[1] + b0); vals.append(mine[idx])
        del Cb, mine
    row, col, val = torch.cat(rows), torch.cat(cols), torch.cat(vals)
    key = row * nc + col
    key, order = torch.sort(key)
    return DCsr(nc, nc, coarse_split, comm.rank, key // nc, key % nc, val[order])


def filter_entries_dist(Ac: DCsr, thre: float) -> DCsr:
    """saena_object::filter on my rows: off-diagonal |v| <= thre is lumped into the diagonal (a row's diagonal lives in
    the row)"""
    n, dev = Ac.m, Ac.val.device
    grow = Ac.row + Ac.r0
    is_diag = grow == Ac.col
    keep = (Ac.val.abs() > thre) | is_diag
    add = torch.zeros(n, dtype=torch.float64, device=dev)
    add.index_add_(0, Ac.row[~keep], Ac.val[~keep])
    row, col, val = Ac.row[keep], Ac.col[keep], Ac.val[keep].clone()
    d = (row + Ac.r0) == col
    val[d] = val[d] + add[row[d]]
    val[d] = torch.where(val[d].abs() < ALMOST_ZERO, torch.ones_like(val[d]), val[d])
    has_diag = torch.zeros(n, dtype=torch.bool, device=dev)
    has_diag[row[d]] = True
    if n and not bool(has_diag.all()):
        miss = torch.nonzero(~has_diag).flatten()
        C = _coalesce(n, Ac.n_cols, torch.cat([row, miss]), torch.cat([col, miss + Ac.r0]),
                      torch.cat([val, torch.ones(miss.numel(), dtype=torch.float64, device=dev)]))
        row, col, val = C.row, C.col, C.val
    return DCsr(Ac.n_rows, Ac.n_cols, Ac.split, Ac.rank, row, col, val)


# ------------------------------------------------------------------------------------------
# a rank's share in the reference layout
# ------------------------------------------------------------------------------------------
def rank_operator(comm: Comm, kind: int, level: int, M: DCsr, col_split: np.ndarray, use_double: bool) -> Operator:
    """sa_setup.rank_layout where every rank holds only its own rows: what the others ask of me arrives through the
    request lists (recvCount -> MPI_Alltoall -> sendCount in set_off_on_diagonal, src/saena_matrix_setup.cpp:904-1072)"""
    def send_side(distinct):
        f = Fetcher(comm, col_split, distinct)
        return f.serve_counts, f.serve_idx

    return rank_layout(kind, level, M.row, M.col, M.val, M.n_rows, M.n_cols, M.split, col_split, comm.rank, use_double,
                       send_side)


# ------------------------------------------------------------------------------------------
# the level loop
# ------------------------------------------------------------------------------------------
def coarsen(comm: Comm, A0: DCsr, opts: SetupOptions, agglomerate_below: int, rebalance_above: float,
            dense: Optional[bool] = None, verbose: bool = False):
    """Collective generator.  A0: my rows of the fine matrix (any row partition; it is moved to the nnz-balanced one).
    Yields every level, finest first, as (DeviceLevel with my rows of A, P and R, so, sn): `so` is the partition R
    writes the coarse vector into (P's column partition), `sn` the one the coarse level lives on; the coarsest level
    comes last, with P, R, so and sn None.  Where a coarse level lives follows hierarchy.partition_hierarchy's rules
    (hierarchy.coarse_placement).  The generator drops its references to a level's tensors once it is resumed."""
    rank, nprocs = comm.rank, comm.world
    say = (lambda s: print(s, file=sys.stderr, flush=True)) if (verbose and rank == 0) else (lambda s: None)

    A = repartition(comm, A0, balanced_split_dist(comm, A0))
    filter_thre, filter_it = opts.filter_thre, 0
    l, last_level = 0, False
    a_use_double = opts.float_level != 0                  # saena_object.cpp:241-244
    while True:
        t_lv = time.perf_counter()
        cm = ColMap(comm, A.split, A.col)
        col_ext = cm.to_ext(A.col)
        d = diag_local(A)
        if comm.sum(int((d.abs() < ALMOST_ZERO).sum())) > 0:
            raise ValueError("zero diagonal element")      # inverse_diag: print + exit in the reference
        inv_diag = 1.0 / d
        eig = lanczos_eig_max_dist(comm, A, cm, col_ext, inv_diag, opts.lanczos_iters, opts.seed + l)
        g_nnz = comm.sum(A.nnz)
        say(f"level {l}: rows {A.n_rows} nnz {g_nnz} ({g_nnz / A.n_rows:.1f}/row) eig {eig:.4f} "
            f"[rows per rank {comm.gather_ints(A.m).tolist()}]")
        lv = DeviceLevel(A=A, inv_diag=inv_diag, eig_max=eig, a_use_double=a_use_double)
        if l >= opts.max_level or last_level:
            yield lv, None, None
            return
        t_ag = time.perf_counter()
        s_r, s_c = strength_graph_dist(A, cm, col_ext, opts.conn_str)
        agg_c_ext, nc, so, rounds = aggregate_dist(comm, cm, s_r, s_c)
        del s_r, s_c
        say(f"   aggregation: {nc} aggregates in {rounds} rounds, {time.perf_counter() - t_ag:.1f}s")
        t_rap = time.perf_counter()
        # find_aggregation's dynamic-level rule: the level about to be created is the last one
        if opts.dynamic_levels:
            last_level = bool(nc <= opts.least_row_threshold or
                              np.float32(nc) / np.float32(A.n_rows) > np.float32(opts.row_reduction_up_thrshld))
        else:
            last_level = (l + 1 == opts.max_level)
        P = prolongator_dist(A, col_ext, agg_c_ext, nc, inv_diag)
        del agg_c_ext
        Ac = galerkin_dist(comm, A, cm, col_ext, P, so, dense=dense)
        del cm, col_ext
        filter_it += 1
        if filter_it >= opts.filter_start:
            filter_thre = min(filter_thre, opts.filter_max)
            Ac = filter_entries_dist(Ac, filter_thre)
            filter_thre *= 10 ** opts.filter_rate

        def imbalance():                 # Ac lives on the aligned split `so`
            per = comm.gather_ints(Ac.nnz)
            return per.max() * nprocs / max(int(per.sum()), 1)

        # a level whose split leaves every row on rank 0 takes its coarse level along; R and P are partitioned by a
        # re-balanced split too
        so, sn, _ = coarse_placement(nprocs, nc, last_level or l + 1 >= opts.max_level, bool(A.split[1] == A.n_rows),
                                     agglomerate_below, rebalance_above, so, imbalance,
                                     lambda: balanced_split_dist(comm, Ac))
        lv.P, lv.R = P, transpose_dist(comm, P, so)
        lv.pr_use_double = not (l >= opts.float_level)     # saena_object.cpp:277-280
        del P
        yield lv, so, sn
        del lv
        A = repartition(comm, Ac, sn)
        del Ac
        say(f"   P, R, RAP, filter, operators: {time.perf_counter() - t_rap:.1f}s (level {time.perf_counter() - t_lv:.1f}s)")
        a_use_double = not (l + 1 >= opts.float_level)     # :281-284
        l += 1


def build_distributed_hierarchy(A0: DCsr, opts: Optional[SetupOptions] = None, agglomerate_below: int = 10_000,
                                rebalance_above: float = 1.10, verbose: bool = False, dense: Optional[bool] = None,
                                comm: Optional[Comm] = None):
    """Collective.  A0: my rows of the fine matrix (any row partition; it is moved to the nnz-balanced one).
    Returns (this rank's Hierarchy, summary lines of the global hierarchy).  Each level is turned into this rank's
    Operators as soon as it is coarsened and its device tensors are dropped, so the setup holds one level at a time."""
    comm = comm or Comm(A0.val.device)
    rank, nprocs = comm.rank, comm.world
    levels: List[Level] = []
    summary = []
    for l, (lv, so, sn) in enumerate(coarsen(comm, A0, opts or SetupOptions(), agglomerate_below, rebalance_above,
                                             dense, verbose)):
        A = lv.A
        g_nnz = comm.sum(A.nnz)
        line = f"L{l}: M={A.n_rows} nnz={g_nnz} ({g_nnz / A.n_rows:.1f}/row) eig={lv.eig_max:.4f}"
        out = Level(level=l, A=rank_operator(comm, KIND_A, l, A, A.split, lv.a_use_double),
                    inv_diag=lv.inv_diag.cpu().numpy(), eig_max=lv.eig_max, active=A.m > 0)
        if lv.P is not None:
            out.P = rank_operator(comm, KIND_P, l, lv.P, so, lv.pr_use_double)
            out.R = rank_operator(comm, KIND_R, l, lv.R, A.split, lv.pr_use_double)
            out.M_coarse_old = int(so[rank + 1] - so[rank])
            out.M_coarse = int(sn[rank + 1] - sn[rank])
            out.repart_send, out.repart_recv = repart_plan(so, sn, rank)
            line += f" | P nnz={comm.sum(lv.P.nnz)}"
        else:
            # the coarsest operator as global COO on every rank (tiny)
            own = A.m > 0 or nprocs == 1
            src = int(np.flatnonzero(np.diff(A.split) > 0)[0]) if A.n_rows else 0
            crow = comm.bcast_tensor((A.row + A.r0) if own else None, torch.int64, src)
            ccol = comm.bcast_tensor(A.col if own else None, torch.int64, src)
            cval = comm.bcast_tensor(A.val if own else None, torch.float64, src)
            coarse = dict(coarse_n=A.n_rows, coarse_row=crow.to(torch.int32).cpu().numpy(),
                          coarse_col=ccol.to(torch.int32).cpu().numpy(), coarse_val=cval.cpu().numpy())
        levels.append(out)
        summary.append(line)
        del lv, A
    return Hierarchy(levels=levels, nprocs=nprocs, rank=rank, **coarse), summary


# ------------------------------------------------------------------------------------------
# the synthetic fine matrix, my rows only
# ------------------------------------------------------------------------------------------
def poisson3d_rows(n: int, r0: int, r1: int, device) -> tuple:
    """rows [r0, r1) of sa_setup.poisson3d_coo(n), sorted row-major: (local row, global col, val)"""
    dev = torch.device(device)
    h2 = float((n + 1) ** 2)
    idx = torch.arange(r0, r1, dtype=torch.int64, device=dev)
    i, j, k = idx % n, (idx // n) % n, idx // (n * n)
    offs = (-n * n, -n, -1, 0, 1, n, n * n)
    oks = (k > 0, j > 0, i > 0, torch.ones_like(i, dtype=torch.bool), i < n - 1, j < n - 1, k < n - 1)
    ok = torch.stack(oks, 1)                                             # [m, 7] in ascending column order
    col = idx[:, None] + torch.tensor(offs, dtype=torch.int64, device=dev)[None, :]
    val = torch.full((7,), -h2, dtype=torch.float64, device=dev)
    val[3] = 6.0 * h2
    row = (idx - r0)[:, None].expand(-1, 7)
    return row[ok], col[ok], val[None, :].expand(idx.numel(), -1)[ok]


def poisson3d_dcsr(n: int, comm: Comm) -> DCsr:
    """the fine 7-point matrix, equal row blocks (build_distributed_hierarchy re-balances by nnz)"""
    N = n ** 3
    split = np.array([N * r // comm.world for r in range(comm.world + 1)], I64)
    row, col, val = poisson3d_rows(n, int(split[comm.rank]), int(split[comm.rank + 1]), comm.dev)
    return DCsr(N, N, split, comm.rank, row, col, val)


def poisson3d_rhs_rows(n: int, r0: int, r1: int) -> np.ndarray:
    """entries [r0, r1) of sa_setup.poisson3d_rhs(n)"""
    import math
    mx = n + 2
    t = np.arange(1, mx - 1, dtype=np.float64) / (mx - 1)
    s = np.sin(2 * math.pi * t)
    idx = np.arange(r0, r1, dtype=np.int64)
    i, j, k = idx % n, (idx // n) % n, idx // (n * n)
    return 12 * math.pi ** 2 * s[i] * s[j] * s[k]


def coo_dcsr(n: int, row, col, val, comm: Comm, split: Optional[np.ndarray] = None) -> DCsr:
    """a global COO (every rank holds all of it: small test inputs) -> my rows of a row partition (equal blocks
    unless `split` is given)"""
    split = np.array([n * r // comm.world for r in range(comm.world + 1)], I64) if split is None else np.asarray(split, I64)
    r0, r1 = int(split[comm.rank]), int(split[comm.rank + 1])
    row, col, val = (np.asarray(row, I64), np.asarray(col, I64), np.asarray(val, F64))
    keep = (row >= r0) & (row < r1)
    C = _coalesce(max(r1 - r0, 1), n, torch.as_tensor(row[keep] - r0, device=comm.dev),
                  torch.as_tensor(col[keep], device=comm.dev), torch.as_tensor(val[keep], device=comm.dev))
    return DCsr(n, n, split, comm.rank, C.row, C.col, C.val)
