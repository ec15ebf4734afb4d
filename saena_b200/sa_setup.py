"""Smoothed-aggregation setup restated with tensor ops -- ONLY to feed the benchmark and the
large-size tests with a hierarchy of the reference's shape.

Why this exists.  The AMG setup is outside this package's scope: it stays on the reference's
host code (BASELINE.json north_star) and the drop-in adaptor uploads whatever
`saena_object::setup` produced.  But the reference's setup cannot feed the bench: measured in
this image it needs 3 s for 30^3 unknowns and 47 s for 64^3 (std::set assembly, recursive
SpGEMM), i.e. the better part of an hour for the 256^3 workload, and its sources do not exist on
the GPU box.  This module and sa_setup_dist.py restate the setup's algorithm with torch tensor ops
(GPU when there is one) so that the bench solves on a hierarchy built by the SAME rules:

  strength of connection   create_strength_matrix   src/saena_object_setup1.cpp:520-720
                           + threshold              src/strength_matrix.cpp:233-270
  aggregation              aggregation_1_dist       src/saena_object_setup1.cpp:724-995
                           (a synchronous, data-parallel iteration: restated round for round,
                            so the aggregates are IDENTICAL to the reference's on one rank)
  coarse numbering         aggregate_index_update   src/saena_object_setup1.cpp:2103-2160
  prolongator              SA(): P = (I - w D^-1 A) P_t, w = float(2/3), drop |v| <= 1e-14
                                                    src/saena_object_setup1.cpp:8-254
  restriction              R = P^T                  src/restrict_matrix.cpp:10-494
  Galerkin product         Ac = R A P               src/saena_object_setup2.cpp:361
  filter                   small entries lumped to the diagonal, threshold x10 per level
                                                    src/saena_object_setup2.cpp:849-891
  level count              dynamic levels           src/saena_object_setup1.cpp:385-392
  Chebyshev bound          1.0001 * lambda_max(D^-1 A) by Lanczos, include/lamlan_saena.h:13-79
                           (the reference starts Lanczos from std::random_device and is not
                            reproducible run to run; here the start vector is seeded)
  precision flags          float_level              src/saena_object.cpp:241-244,277-285

The steps and the level loop are written once, row-partitioned over the ranks, in sa_setup_dist.py.
`build_device_hierarchy` runs that loop on one rank, where a rank's rows are the whole matrix and
every exchange is empty, and keeps the global hierarchy on the device; `DeviceHierarchy.to_rank`
cuts any rank's share out of it.  This module holds the sparse-matrix primitives both use, the
reference layout of a rank's operator and the synthetic inputs.

tests/test_sa_setup.py checks the result against the reference's own hierarchy (same
aggregates / same operators to rounding) where oracle/_ref is available.  torch here is
plumbing for the setup only; nothing in the solve path imports this module.
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass
from typing import List, Optional

import numpy as np
import torch

from .hierarchy import (KIND_A, KIND_P, KIND_R, Hierarchy, Level, Operator, balanced_split, coarse_placement,
                        csr_from_counts, repart_plan, split_imbalance)

ALMOST_ZERO = 1e-14                  # include/data_struct.h:41
JACOBI_OMEGA = float(np.float32(2.0 / 3))   # saena_matrix.h:182 (a float, promoted)
BIG = 2 ** 62


@dataclass
class SetupOptions:
    """data/options006_poisson.xml"""
    conn_str: float = 0.2
    dynamic_levels: bool = True
    max_level: int = 20
    float_level: int = 0
    filter_thre: float = 1e-12
    filter_max: float = 1e-9
    filter_start: int = 1
    filter_rate: int = 1
    least_row_threshold: int = 100           # saena_object.h:43
    row_reduction_up_thrshld: float = 0.90   # saena_object.h:46
    lanczos_iters: int = 20
    seed: int = 2024


class _Csr:
    """row-major sorted COO/CSR triple on one torch device"""

    def __init__(self, n_rows, n_cols, row, col, val):
        self.n_rows, self.n_cols, self.row, self.col, self.val = n_rows, n_cols, row, col, val

    @property
    def nnz(self):
        return int(self.val.numel())

    def counts(self):
        return torch.bincount(self.row, minlength=self.n_rows)


def _coalesce(n_rows, n_cols, row, col, val) -> _Csr:
    """sort by (row, col) and add duplicates"""
    key = row * n_cols + col
    key, order = torch.sort(key)
    val = val[order]
    uk, inv = torch.unique_consecutive(key, return_inverse=True)
    out = torch.zeros(uk.numel(), dtype=torch.float64, device=val.device)
    out.index_add_(0, inv, val)
    return _Csr(n_rows, n_cols, uk // n_cols, uk % n_cols, out)


# The setup on one rank routes its products through the library's device SpGEMM since it passed
# tests/test_zzz_spgemm_gpu.py on a B200 (scipy, the reference's golden hierarchies, the live reference at 32^3, route
# equality at 64^3) and built the 256^3 bench hierarchy end to end (profiles/r02_setup_time.json,
# r02_bench_n1_native_spgemm.json).  Several ranks keep the tensor-op route until their own run with the device
# SpGEMM (SAENA_SETUP_SPGEMM=native asks for it there too).
def _native_spgemm_enabled(dev, world: int) -> bool:
    """SAENA_SETUP_SPGEMM=native: the library's own SpGEMM (csrc/spgemm.cu, SURVEY 8f #3) does the products on a CUDA
    device; =torch: the tensor-op route below (the CPU path, and the A/B).  The default depends on the number of
    ranks only, so every rank takes the same route."""
    default = "native" if world == 1 else "torch"
    return dev.type == "cuda" and os.environ.get("SAENA_SETUP_SPGEMM", default) != "torch"


def _spgemm_native(A: _Csr, B: _Csr) -> _Csr:
    """C = A B with the hand-written device kernels of libsaena_b200.so (saena_b200_spgemm_symbolic / _numeric)"""
    from . import native
    dev = A.val.device

    def csr_arrays(M: _Csr):
        rp = torch.zeros(M.n_rows + 1, dtype=torch.int64, device=dev)
        rp[1:] = torch.cumsum(M.counts(), 0)
        return rp, M.col.to(torch.int32).contiguous(), M.val.contiguous()

    a_rp, a_col, a_val = csr_arrays(A)
    b_rp, b_col, b_val = csr_arrays(B)
    c_rp, c_col, c_val = native.spgemm_csr(A.n_rows, A.n_cols, B.n_cols, a_rp, a_col, a_val, b_rp, b_col, b_val)
    row = torch.repeat_interleave(torch.arange(A.n_rows, device=dev), c_rp[1:] - c_rp[:-1])
    return _Csr(A.n_rows, B.n_cols, row, c_col.to(torch.int64), c_val)


def _spgemm(A: _Csr, B: _Csr, chunk_products: int, native: bool) -> _Csr:
    """C = A B: the library's device SpGEMM if `native` (_native_spgemm_enabled); otherwise expand / sort / compress
    with tensor ops, in row chunks bounded by the number of products"""
    dev = A.val.device
    if native and A.n_rows < 2 ** 31 and B.n_cols < 2 ** 31 - 1:
        return _spgemm_native(A, B)
    b_counts = B.counts()
    b_ptr = torch.zeros(B.n_rows + 1, dtype=torch.int64, device=dev)
    b_ptr[1:] = torch.cumsum(b_counts, 0)
    per_entry = b_counts[A.col]                       # products each A entry generates
    a_counts = A.counts()
    a_ptr = torch.zeros(A.n_rows + 1, dtype=torch.int64, device=dev)
    a_ptr[1:] = torch.cumsum(a_counts, 0)
    prod_cum = torch.zeros(A.nnz + 1, dtype=torch.int64, device=dev)
    prod_cum[1:] = torch.cumsum(per_entry, 0)
    rows_out, cols_out, vals_out = [], [], []
    r0 = 0
    row_prod_cum = prod_cum[a_ptr]                    # products before each row
    total = int(prod_cum[-1])
    while r0 < A.n_rows:
        # largest r1 with products(r0..r1) <= chunk
        target = int(row_prod_cum[r0]) + chunk_products
        r1 = int(torch.searchsorted(row_prod_cum, torch.tensor([target], device=dev), right=True)[0]) - 1
        r1 = max(r1, r0 + 1)
        r1 = min(r1, A.n_rows)
        e0, e1 = int(a_ptr[r0]), int(a_ptr[r1])
        if e1 > e0:
            pe = per_entry[e0:e1]
            n_prod = int(pe.sum())
            if n_prod:
                src = torch.repeat_interleave(torch.arange(e0, e1, device=dev), pe)      # A entry of each product
                first = prod_cum[e0:e1] - prod_cum[e0]
                within = torch.arange(n_prod, device=dev) - torch.repeat_interleave(first, pe)
                bidx = b_ptr[A.col[src]] + within
                c = _coalesce(A.n_rows, B.n_cols, A.row[src], B.col[bidx], A.val[src] * B.val[bidx])
                rows_out.append(c.row); cols_out.append(c.col); vals_out.append(c.val)
        r0 = r1
    del total
    if not rows_out:
        z = torch.zeros(0, dtype=torch.int64, device=dev)
        return _Csr(A.n_rows, B.n_cols, z, z.clone(), torch.zeros(0, dtype=torch.float64, device=dev))
    return _Csr(A.n_rows, B.n_cols, torch.cat(rows_out), torch.cat(cols_out), torch.cat(vals_out))


def _to_torch_csr(A: _Csr) -> torch.Tensor:
    crow = torch.zeros(A.n_rows + 1, dtype=torch.int64, device=A.val.device)
    crow[1:] = torch.cumsum(A.counts(), 0)
    return torch.sparse_csr_tensor(crow, A.col, A.val, size=(A.n_rows, A.n_cols))


def _transpose(A: _Csr) -> _Csr:
    key = A.col * A.n_rows + A.row
    key, order = torch.sort(key)
    return _Csr(A.n_cols, A.n_rows, key // A.n_rows, key % A.n_rows, A.val[order])


# ------------------------------------------------------------------------------------------
def _expand_segments(ptr: torch.Tensor, rows: torch.Tensor):
    """entry indices of the CSR segments of `rows` and, per entry, the position of its row in `rows`"""
    dev = rows.device
    start = ptr[rows]
    deg = ptr[rows + 1] - start
    total = int(deg.sum())
    seg = torch.repeat_interleave(torch.arange(rows.numel(), device=dev), deg, output_size=total)
    first = torch.cumsum(deg, 0) - deg
    e = start[seg] + (torch.arange(total, device=dev) - first[seg])
    return e, seg


# ------------------------------------------------------------------------------------------
@dataclass
class DeviceLevel:
    """one level of the setup as torch tensors: this rank's rows of A, P and R (sa_setup_dist.DCsr; on one rank the
    global matrices)"""
    A: "DCsr"
    inv_diag: torch.Tensor
    eig_max: float
    a_use_double: bool
    P: Optional["DCsr"] = None
    R: Optional["DCsr"] = None
    pr_use_double: bool = True


def rank_layout(kind, level, row, col, val, Mbig, Nbig, row_split, col_split, rank, use_double, send_side) -> Operator:
    """One rank's Operator from its rows (`row` local ids, `col` global ids, row-major sorted), on device tensors: the
    receive half of hierarchy.split_operator -- the local block, the remote block column-major and grouped by owner.
    The send half is what the other ranks ask of this one, which the builders learn in different ways:
    send_side(distinct remote columns of this rank) -> (entries sent to each rank, their local column ids)."""
    dev = val.device
    nprocs = len(col_split) - 1
    r0, nrows = int(row_split[rank]), int(row_split[rank + 1] - row_split[rank])
    c0, c1 = int(col_split[rank]), int(col_split[rank + 1])
    local = (col >= c0) & (col < c1)
    op = dict(kind=kind, level=level, M=nrows, Mbig=Mbig, Nbig=Nbig, row_offset=r0, col_offset=c0,
              n_local_cols=c1 - c0, use_double=use_double, nprocs=nprocs, rank=rank)
    op["nnzPerRow_local"] = torch.bincount(row[local], minlength=nrows).to(torch.int32).cpu().numpy()
    op["col_local"] = col[local].to(torch.int32).cpu().numpy()
    op["val_local"] = val[local].cpu().numpy()
    if nprocs == 1:
        return Operator(**op)
    # remote part: column-major (col, then row)
    rr, rc, rv = row[~local], col[~local], val[~local]
    order = torch.argsort(rc * max(nrows, 1) + rr)
    rr, rc, rv = rr[order], rc[order], rv[order]
    distinct, counts = torch.unique_consecutive(rc, return_counts=True)
    cs = torch.as_tensor(np.asarray(col_split, np.int64), device=dev)
    owner_d = torch.searchsorted(cs, distinct, right=True) - 1
    owner_e = torch.searchsorted(cs, rc, right=True) - 1
    recv_count = torch.bincount(owner_d, minlength=nprocs).cpu().numpy().astype(np.int32)
    nnz_per_proc = torch.bincount(owner_e, minlength=nprocs).cpu().numpy()
    op["row_remote"] = rr.to(torch.int32).cpu().numpy()
    op["val_remote"] = rv.cpu().numpy()
    op["nnzPerCol_remote"] = counts.to(torch.int32).cpu().numpy()
    op["nnzPerProcScan"] = np.concatenate(([0], np.cumsum(nnz_per_proc))).astype(np.int64)
    op["rdispls"] = np.concatenate(([0], np.cumsum(recv_count)[:-1])).astype(np.int32)
    op["recvProcRank"] = np.flatnonzero(recv_count).astype(np.int32)
    op["recvProcCount"] = recv_count[recv_count != 0]
    send_count, v_index = send_side(distinct)
    send_count = np.asarray(send_count, np.int32)
    op["vIndex"] = v_index.to(torch.int32).cpu().numpy()
    op["vdispls"] = np.concatenate(([0], np.cumsum(send_count)[:-1])).astype(np.int32)
    op["sendProcRank"] = np.flatnonzero(send_count).astype(np.int32)
    op["sendProcCount"] = send_count[send_count != 0]
    return Operator(**op)


class DeviceHierarchy:
    """The global (one-rank) hierarchy as torch tensors, plus its conversion to any rank's share
    of a 1-D row partition in the reference layout (`saena_b200.hierarchy.Operator`)."""

    def __init__(self, levels: List[DeviceLevel]):
        self.levels = levels

    def summary(self) -> str:
        return "\n".join(f"L{l}: M={lv.A.n_rows} nnz={lv.A.nnz} ({lv.A.nnz / lv.A.n_rows:.1f}/row) eig={lv.eig_max:.4f}"
                         + (f" | P nnz={lv.P.nnz}" if lv.P is not None else "") for l, lv in enumerate(self.levels))

    # -- partitions ----------------------------------------------------------------------------
    @staticmethod
    def _balanced_split(M, nprocs: int) -> np.ndarray:
        """nnz-balanced contiguous row blocks (hierarchy.balanced_split on device counts)"""
        return balanced_split(csr_from_counts(M.counts().cpu().numpy()), nprocs).astype(np.int64)

    @staticmethod
    def _aligned_coarse_split(R, fine_split: np.ndarray) -> np.ndarray:
        """hierarchy.aligned_coarse_split on device tensors"""
        dev = R.val.device
        nprocs = len(fine_split) - 1
        nc = R.n_rows
        a = R.val.abs()
        row_max = torch.zeros(nc, dtype=torch.float64, device=dev)
        row_max.scatter_reduce_(0, R.row, a, reduce="amax", include_self=False)
        cand = torch.where(a == row_max[R.row], R.col, torch.full_like(R.col, BIG))
        arg_col = torch.full((nc,), BIG, dtype=torch.int64, device=dev)
        arg_col.scatter_reduce_(0, R.row, cand, reduce="amin")
        fs = torch.as_tensor(np.asarray(fine_split, np.int64), device=dev)
        owner = torch.clamp(torch.searchsorted(fs, arg_col, right=True) - 1, 0, nprocs - 1)
        owner = torch.cummax(owner, 0).values
        return torch.searchsorted(owner, torch.arange(nprocs + 1, device=dev), right=False).cpu().numpy().astype(np.int64)

    def splits(self, nprocs: int, agglomerate_below: int, rebalance_above: float = 0.0):
        """(row partition of every level, partition R of the level above writes into, agglomerated?)
        -- hierarchy.partition_hierarchy's rules"""
        L = len(self.levels)
        splits, aligned, agglomerated = [self._balanced_split(self.levels[0].A, nprocs)], [None], [False]
        for l in range(1, L):
            A = self.levels[l].A
            follow = self._aligned_coarse_split(self.levels[l - 1].R, splits[-1])
            al, sp, agg = coarse_placement(
                nprocs, A.n_rows, l == L - 1, agglomerated[-1], agglomerate_below, rebalance_above, follow,
                imbalance=lambda: split_imbalance(csr_from_counts(A.counts().cpu().numpy()), follow),
                balanced=lambda: self._balanced_split(A, nprocs))
            aligned.append(al)
            splits.append(sp)
            agglomerated.append(agg)
        return splits, aligned, agglomerated

    @staticmethod
    def _rank_operator(kind, level, M, row_split, col_split, rank, use_double) -> Operator:
        """one rank's Operator -- hierarchy.split_operator restated on device tensors, building
        only `rank`'s arrays (the other ranks' requests are still needed for the send plan)"""
        nprocs = len(row_split) - 1
        r0, r1, c0, c1 = int(row_split[rank]), int(row_split[rank + 1]), int(col_split[rank]), int(col_split[rank + 1])
        mine = (M.row >= r0) & (M.row < r1)

        def send_side(_):
            # what the others ask of me: entries whose column I own and whose row I do not
            rs = torch.as_tensor(row_split, device=M.val.device)
            wanted = (M.col >= c0) & (M.col < c1) & ~mine
            dst = torch.searchsorted(rs, M.row[wanted], right=True) - 1
            key = torch.unique(dst * M.n_cols + M.col[wanted])
            return torch.bincount(key // M.n_cols, minlength=nprocs).cpu().numpy(), key % M.n_cols - c0

        return rank_layout(kind, level, M.row[mine] - r0, M.col[mine], M.val[mine], M.n_rows, M.n_cols, row_split,
                           col_split, rank, use_double, send_side)

    def to_rank(self, rank: int = 0, nprocs: int = 1, agglomerate_below: int = 0,
                rebalance_above: float = 0.0) -> Hierarchy:
        """This rank's share (hierarchy.partition_hierarchy semantics: nnz-balanced row blocks per
        level, levels below `agglomerate_below` global rows -- and always the coarsest -- on rank 0)."""
        splits, aligned, agglomerated = self.splits(nprocs, agglomerate_below, rebalance_above)
        levels = []
        for l, lv in enumerate(self.levels):
            sp = splits[l]
            r0, r1 = int(sp[rank]), int(sp[rank + 1])
            A = self._rank_operator(KIND_A, l, lv.A, sp, sp, rank, lv.a_use_double)
            out = Level(level=l, A=A, inv_diag=lv.inv_diag[r0:r1].cpu().numpy(), eig_max=lv.eig_max, active=r1 > r0)
            if lv.P is not None:
                so, sn = aligned[l + 1], splits[l + 1]
                out.P = self._rank_operator(KIND_P, l, lv.P, sp, so, rank, lv.pr_use_double)
                out.R = self._rank_operator(KIND_R, l, lv.R, so, sp, rank, lv.pr_use_double)
                out.M_coarse_old = int(so[rank + 1] - so[rank])
                out.M_coarse = int(sn[rank + 1] - sn[rank])
                out.repart_send, out.repart_recv = repart_plan(so, sn, rank)
            levels.append(out)
        last = self.levels[-1].A
        return Hierarchy(levels=levels, coarse_n=last.n_rows, coarse_row=last.row.to(torch.int32).cpu().numpy(),
                         coarse_col=last.col.to(torch.int32).cpu().numpy(), coarse_val=last.val.cpu().numpy(),
                         nprocs=nprocs, rank=rank)


def build_device_hierarchy(n: int, row, col, val, opts: Optional[SetupOptions] = None, device: Optional[str] = None,
                           verbose: bool = False) -> DeviceHierarchy:
    """Global hierarchy from a square matrix given as COO (any order, duplicates added): the coarsening loop of
    sa_setup_dist.py on one rank, where this rank's rows are the whole matrix."""
    from . import sa_setup_dist as sd
    dev = torch.device(device or ("cuda" if torch.cuda.is_available() else "cpu"))

    def as_t(a, dt):
        return a.to(dev, dt) if isinstance(a, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(a), device=dev).to(dt)

    A = _coalesce(n, n, as_t(row, torch.int64), as_t(col, torch.int64), as_t(val, torch.float64))
    A0 = sd.DCsr(n, n, [0, n], 0, A.row, A.col, A.val)
    del A
    levels = sd.coarsen(sd.Comm(dev, one_rank=True), A0, opts or SetupOptions(), 0, 0.0, verbose=verbose)
    return DeviceHierarchy([lv for lv, _, _ in levels])


def build_hierarchy(n: int, row, col, val, opts: Optional[SetupOptions] = None, device: Optional[str] = None,
                    verbose: bool = False) -> Hierarchy:
    """One-rank hierarchy in the reference layout."""
    return build_device_hierarchy(n, row, col, val, opts, device, verbose).to_rank(0, 1)


# ------------------------------------------------------------------------------------------
# the synthetic inputs of SURVEY.md 8d
# ------------------------------------------------------------------------------------------
def poisson3d_coo(n: int):
    """7-point Laplacian on the n^3 INTERIOR nodes of an (n+2)^3 grid: what laplacian3D(mx = n+2) +
    set_remove_boundary(true) leaves (src/aux_functions2.cpp:326-365): diag 6/h^2, off-diag -1/h^2,
    h = 1/(mx-1)."""
    mx = n + 2
    h2 = float((mx - 1) ** 2)
    idx = np.arange(n ** 3, dtype=np.int64)
    i, j, k = idx % n, (idx // n) % n, idx // (n * n)
    rows, cols, vals = [idx], [idx], [np.full(idx.shape, 6.0 * h2)]
    for ok, off in ((i > 0, -1), (i < n - 1, 1), (j > 0, -n), (j < n - 1, n), (k > 0, -n * n), (k < n - 1, n * n)):
        rows.append(idx[ok]); cols.append(idx[ok] + off); vals.append(np.full(int(ok.sum()), -h2))
    return n ** 3, np.concatenate(rows), np.concatenate(cols), np.concatenate(vals)


def convdiff3d_coo(n: int, wind=(1.0, 0.5, 0.25), peclet: float = 20.0):
    """Nonsymmetric 7-point convection-diffusion operator -lap(u) + b . grad(u) on the n^3 interior nodes of the unit
    cube, b = peclet * wind, first-order upwind differences for the convection term: diag 6/h^2 + sum|b|/h, neighbour
    -1/h^2, and -|b_d|/h more on the upstream neighbour of each direction d, h = 1/(n+1).  An M-matrix, not
    symmetric (the GMRES solve's test and measurement input)."""
    h = 1.0 / (n + 1)
    b = peclet * np.asarray(wind, np.float64)
    idx = np.arange(n ** 3, dtype=np.int64)
    coord = (idx % n, (idx // n) % n, idx // (n * n))
    rows, cols, vals = [idx], [idx], [np.full(idx.shape, 6.0 / h ** 2 + np.abs(b).sum() / h)]
    for d, stride in enumerate((1, n, n * n)):
        for s in (-1, 1):
            ok = coord[d] > 0 if s < 0 else coord[d] < n - 1
            upstream = (b[d] > 0) == (s < 0)
            v = -1.0 / h ** 2 - (abs(b[d]) / h if upstream else 0.0)
            rows.append(idx[ok]); cols.append(idx[ok] + s * stride); vals.append(np.full(int(ok.sum()), v))
    return n ** 3, np.concatenate(rows), np.concatenate(cols), np.concatenate(vals)


def poisson3d_rhs(n: int) -> np.ndarray:
    """laplacian3D_set_rhs restricted to interior nodes (src/aux_functions2.cpp:629-700):
    12 pi^2 sin(2 pi x) sin(2 pi y) sin(2 pi z) at x = i/(mx-1)"""
    mx = n + 2
    t = np.arange(1, mx - 1, dtype=np.float64) / (mx - 1)
    s = np.sin(2 * math.pi * t)
    return (12 * math.pi ** 2 * s[None, None, :] * s[None, :, None] * s[:, None, None]).ravel()


# forward half of a 2-D neighbourhood ordered by distance: node (x, y) couples to (x+dx, y+dy); the
# mirrored entries make the pattern symmetric
_HALF_OFFSETS = [(1, 0), (0, 1), (1, 1), (-1, 1), (2, 0), (0, 2), (2, 1), (1, 2), (-1, 2), (-2, 1), (2, 2), (-2, 2),
                 (3, 0), (0, 3), (3, 1), (1, 3), (-1, 3), (-3, 1), (3, 2), (2, 3), (-2, 3), (-3, 2), (4, 0), (0, 4)]


def unstructured2d_coo(g: int, seed: int = 2024, row_lengths=(6, 8, 10), weights=(16, 48, 20), tile: int = 16,
                       shift: float = 0.05):
    """Synthetic 2-D Helmholtz-like matrix with an unstructured-mesh pattern (BASELINE.json configs[4],
    SURVEY.md 8d): g*g nodes; the number of entries per row is drawn from the empirical distribution of
    the shape donors data/Helmholtz2D_CG_curved_tri/*.mtx (P2: 6/8/10 entries in proportion 16:48:20;
    pass row_lengths=(24, 32, 40) for the P8 shape); every node couples to its nearest neighbours until
    its drawn length is reached, the pattern is then symmetrised; nodes are numbered tile by tile
    with a random order inside each `tile` x `tile` patch (mesh-generator-like locality, irregular
    gathers); off-diagonals -(0.5 + u), u uniform, symmetric; diagonal = sum |off-diagonal| * (1 + shift):
    SPD, the positive shift being the Helmholtz term.  Returns (n, row, col, val) with duplicates-free COO."""
    rng = np.random.default_rng(seed)
    n = g * g
    x, y = np.meshgrid(np.arange(g), np.arange(g), indexing="xy")
    x, y = x.ravel(), y.ravel()
    # numbering: tiles in row-major order, random order inside a tile
    tx, ty = x // tile, y // tile
    key = (ty * ((g + tile - 1) // tile) + tx).astype(np.int64) * (tile * tile * 4) + rng.permutation(n) % (tile * tile * 4)
    order = np.argsort(key, kind="stable")
    number = np.empty(n, np.int64)
    number[order] = np.arange(n)
    # forward edges until the drawn row length is reached (half of the off-diagonal count each way)
    want = rng.choice(np.asarray(row_lengths), size=n, p=np.asarray(weights, float) / np.sum(weights))
    half = (want - 1 + 1) // 2
    src, dst = [], []
    for k, (dx, dy) in enumerate(_HALF_OFFSETS[:int(half.max())]):
        ok = (half > k) & (x + dx >= 0) & (x + dx < g) & (y + dy < g)
        src.append(np.flatnonzero(ok))
        dst.append(src[-1] + dx + dy * g)
    src, dst = np.concatenate(src), np.concatenate(dst)
    w = -(0.5 + rng.uniform(0, 1, len(src)))
    i, j = number[src], number[dst]
    diag = np.zeros(n)
    np.add.at(diag, i, -w)
    np.add.at(diag, j, -w)
    diag *= 1.0 + shift
    diag[diag == 0] = 1.0
    row = np.concatenate((i, j, np.arange(n)))
    col = np.concatenate((j, i, np.arange(n)))
    val = np.concatenate((w, w, diag))
    return n, row, col, val


def unstructured2d_rhs(n: int, seed: int = 2024) -> np.ndarray:
    return np.random.default_rng(seed + 1).uniform(-1, 1, n)
