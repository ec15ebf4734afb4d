"""Host-side containers for a finished AMG hierarchy in the reference's operator layout.

The AMG *setup* is not part of this package (it stays on the reference's host code, see
DESIGN.md).  What the solve path needs is the layout the reference's setup leaves behind --
the arrays `saena_matrix::set_off_on_diagonal` builds
(/root/reference/src/saena_matrix_setup.cpp:793-1098) and its twins
`prolong_matrix::findLocalRemote` (/root/reference/src/prolong_matrix.cpp:18-378) and
`restrict_matrix::transposeP` (/root/reference/src/restrict_matrix.cpp:229-494).
`Operator` holds exactly those arrays for one rank (same names, same meaning) and is what
`saena_b200_upload_operator` (include/saena_b200.h) takes.

`split_operator` builds that layout for every rank of a 1-D row partition from a global CSR
matrix.  It restates the splitting loop of set_off_on_diagonal (:827-861: local = columns this
rank owns, re-sorted row-major with GLOBAL column ids; remote = other ranks' columns kept
column-major and grouped by owner) and the plan construction (:904-1072: recvCount ->
Alltoall -> sendCount, vdispls/rdispls, vIndex = requested columns minus split[rank]).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

KIND_A, KIND_P, KIND_R = 0, 1, 2
KIND_NAMES = {KIND_A: "A", KIND_P: "P", KIND_R: "R"}

I32 = np.int32
I64 = np.int64
F64 = np.float64


def _i32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=I32)


def _f64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=F64)


@dataclass
class Operator:
    """One rank's share of A, P or R, in the reference layout (saena_matrix.h:105-149)."""

    kind: int
    level: int
    M: int                      # local rows
    Mbig: int                   # global rows
    Nbig: int                   # global columns
    row_offset: int             # split_rows[rank]
    col_offset: int             # split_cols[rank]; kernels index v - col_offset (saena_matrix_matvec.cpp:56)
    n_local_cols: int           # split_cols[rank+1] - split_cols[rank] == length of the local input vector
    nnzPerRow_local: np.ndarray  # int32[M]
    col_local: np.ndarray        # int32[nnz_local]  GLOBAL column ids, row-major
    val_local: np.ndarray        # float64[nnz_local]
    row_remote: np.ndarray = field(default_factory=lambda: np.zeros(0, I32))        # int32[nnz_remote] local row
    val_remote: np.ndarray = field(default_factory=lambda: np.zeros(0, F64))        # float64[nnz_remote]
    nnzPerCol_remote: np.ndarray = field(default_factory=lambda: np.zeros(0, I32))  # int32[col_remote_size]
    nnzPerProcScan: np.ndarray = field(default_factory=lambda: np.zeros(2, I64))    # int64[nprocs+1]
    vIndex: np.ndarray = field(default_factory=lambda: np.zeros(0, I32))            # int32[vIndexSize] local ids to send
    vdispls: np.ndarray = field(default_factory=lambda: np.zeros(1, I32))           # int32[nprocs]
    rdispls: np.ndarray = field(default_factory=lambda: np.zeros(1, I32))           # int32[nprocs]
    sendProcRank: np.ndarray = field(default_factory=lambda: np.zeros(0, I32))
    sendProcCount: np.ndarray = field(default_factory=lambda: np.zeros(0, I32))
    recvProcRank: np.ndarray = field(default_factory=lambda: np.zeros(0, I32))
    recvProcCount: np.ndarray = field(default_factory=lambda: np.zeros(0, I32))
    use_double: bool = True      # False: ghost values travel as float (matvec_sparse_float)
    # saena_matrix::use_dense (A only; set by the setup when switch_to_dense is on, density > dense_thre and
    # Mbig <= dense_sz_thre, src/saena_object_setup2.cpp:328-329): the reference applies the operator through
    # saena_matrix_dense (src/saena_matrix_dense.cpp:181-340).  Same matrix, same product -- except that with
    # use_double false the dense path casts the WHOLE input vector to float, the rank's own part included (:281).
    use_dense: bool = False
    nprocs: int = 1
    rank: int = 0

    @property
    def nnz_local(self) -> int:
        return int(self.col_local.shape[0])

    @property
    def nnz_remote(self) -> int:
        return int(self.row_remote.shape[0])

    @property
    def col_remote_size(self) -> int:
        return int(self.nnzPerCol_remote.shape[0])

    @property
    def vIndexSize(self) -> int:
        return int(self.vIndex.shape[0])

    @property
    def recvSize(self) -> int:
        return int(self.nnzPerCol_remote.shape[0])

    @property
    def nnz(self) -> int:
        return self.nnz_local + self.nnz_remote

    def to_scipy_local(self):
        """Local block as scipy CSR with LOCAL column ids (host-side convenience for tests)."""
        import scipy.sparse as sp

        indptr = np.zeros(self.M + 1, I64)
        np.cumsum(self.nnzPerRow_local, out=indptr[1:])
        return sp.csr_matrix((self.val_local, self.col_local - self.col_offset, indptr),
                             shape=(self.M, self.n_local_cols))


@dataclass
class Level:
    """grids[l] of the reference (include/grid.h:11-78) restricted to what the solve reads."""

    level: int
    A: Operator
    inv_diag: np.ndarray                 # float64[A.M]   saena_matrix::inv_diag
    eig_max: float                       # saena_matrix::eig_max_of_invdiagXA
    P: Optional[Operator] = None         # None on the coarsest level
    R: Optional[Operator] = None
    active: bool = True                  # saena_matrix::active on this rank
    # Grid::repart_u plan (grid.cpp:3-97): move the coarse vector R produced (partition
    # Ac.split_old) to the partition the coarse grid lives on (Ac.split).  Empty == identity.
    M_coarse_old: int = 0                # Ac.M_old : length of res_coarse as R produces it
    M_coarse: int = 0                    # Ac.M     : length of the coarse grid's vectors on this rank
    repart_send: List[tuple] = field(default_factory=list)  # (peer, offset_in_old, count)
    repart_recv: List[tuple] = field(default_factory=list)  # (peer, offset_in_new, count)
    # D^-1/2 of this level's operator before it was scaled (saena_matrix::inv_sq_diag_orig); only
    # when the hierarchy was set up with scale=true (saena_object_solve.cpp:1245-1247,1264-1266,2709-2711)
    inv_sq_diag: Optional[np.ndarray] = None


@dataclass
class Hierarchy:
    """What `saena_object::setup` leaves in `grids` + the coarsest matrix (one rank's view)."""

    levels: List[Level]
    # coarsest operator gathered as global COO (the reference hands it to SuperLU_DIST,
    # saena_object_solve.cpp:282-308); every rank that takes part in the coarsest solve holds it.
    coarse_n: int = 0
    coarse_row: np.ndarray = field(default_factory=lambda: np.zeros(0, I32))
    coarse_col: np.ndarray = field(default_factory=lambda: np.zeros(0, I32))
    coarse_val: np.ndarray = field(default_factory=lambda: np.zeros(0, F64))
    nprocs: int = 1
    rank: int = 0
    scale: bool = False   # saena_object::scale

    @property
    def max_level(self) -> int:
        return len(self.levels) - 1

    def summary(self) -> str:
        lines = []
        for lv in self.levels:
            s = f"L{lv.level}: M={lv.A.M} nnz={lv.A.nnz} ({lv.A.nnz / max(lv.A.M, 1):.1f}/row) eig={lv.eig_max:.4f}"
            if lv.P is not None:
                s += f" | P nnz={lv.P.nnz} R nnz={lv.R.nnz}"
            lines.append(s)
        return "\n".join(lines)


# --------------------------------------------------------------------------------------
# row partitioning
# --------------------------------------------------------------------------------------
def csr_from_counts(nnz_per_row: np.ndarray) -> np.ndarray:
    indptr = np.zeros(len(nnz_per_row) + 1, I64)
    np.cumsum(nnz_per_row, out=indptr[1:])
    return indptr


def balanced_split(indptr: np.ndarray, nprocs: int) -> np.ndarray:
    """nnz-balanced contiguous row blocks (the goal of repartition_nnz_initial,
    /root/reference/src/saena_matrix_repart.cpp:150-170): rank r gets the rows whose running
    nnz count falls in [r, r+1) * nnz/nprocs."""
    n = len(indptr) - 1
    nnz = int(indptr[-1])
    targets = (np.arange(1, nprocs, dtype=np.float64) * nnz / nprocs)
    cuts = np.searchsorted(indptr[1:], targets, side="left") + 1
    split = np.concatenate(([0], np.minimum(cuts, n), [n])).astype(I64)
    return np.maximum.accumulate(split).astype(I32)


def aligned_coarse_split(r_indptr: np.ndarray, r_indices: np.ndarray, r_data: np.ndarray,
                         fine_split: Sequence[int]) -> np.ndarray:
    """Coarse row partition that follows the fine one: coarse row c goes to the rank that owns the
    fine column carrying its largest |R[c, :]| entry (the aggregate's own nodes), made monotone.
    This is the reference's rule -- an aggregate lives where its root lives, splitNew in
    aggregate_index_update, /root/reference/src/saena_object_setup1.cpp:2124-2132 -- recovered from
    R alone; it keeps the transfer operators' remote parts thin."""
    fine_split = np.asarray(fine_split, I64)
    nprocs = len(fine_split) - 1
    nc = len(r_indptr) - 1
    if nc == 0:
        return np.zeros(nprocs + 1, I64)
    starts = np.asarray(r_indptr[:-1], I64)
    if np.any(np.diff(r_indptr) == 0):
        raise ValueError("restriction operator with an empty row")
    a = np.abs(np.asarray(r_data, F64))
    row_max = np.maximum.reduceat(a, starts)
    rows = np.repeat(np.arange(nc, dtype=I64), np.diff(r_indptr))
    cand = np.where(a == row_max[rows], np.asarray(r_indices, I64), np.iinfo(I64).max)
    arg_col = np.minimum.reduceat(cand, starts)
    owner = np.searchsorted(fine_split, arg_col, side="right") - 1
    owner = np.maximum.accumulate(np.clip(owner, 0, nprocs - 1))
    return np.searchsorted(owner, np.arange(nprocs + 1), side="left").astype(I64)


def split_operator(kind: int, level: int, indptr: np.ndarray, indices: np.ndarray, data: np.ndarray,
                   n_cols: int, row_split: Sequence[int], col_split: Sequence[int],
                   use_double: bool = True) -> List[Operator]:
    """Build every rank's `Operator` from a global CSR matrix (rows sorted, columns ascending
    inside a row) and the 1-D partitions of its rows and columns."""
    row_split = np.asarray(row_split, I64)
    col_split = np.asarray(col_split, I64)
    nprocs = len(row_split) - 1
    n_rows = len(indptr) - 1
    ops: List[Operator] = []
    # what each rank asks of each owner: requested[receiver][owner] = sorted distinct global cols
    requested = [[None] * nprocs for _ in range(nprocs)]
    per_rank = []
    for r in range(nprocs):
        r0, r1 = int(row_split[r]), int(row_split[r + 1])
        M = r1 - r0
        lo, hi = int(indptr[r0]), int(indptr[r1])
        cols = np.asarray(indices[lo:hi], I64)
        vals = np.asarray(data[lo:hi], F64)
        counts = np.diff(indptr[r0:r1 + 1]).astype(I64)
        rows = np.repeat(np.arange(M, dtype=I64), counts)
        c0, c1 = int(col_split[r]), int(col_split[r + 1])
        is_local = (cols >= c0) & (cols < c1)
        # local part: row-major, global column ids (set_off_on_diagonal :833-838, :873)
        nnzPerRow_local = np.bincount(rows[is_local], minlength=M).astype(I32) if M else np.zeros(0, I32)
        col_local = cols[is_local].astype(I32)
        val_local = vals[is_local]
        # remote part: column-major (col, then row), grouped by owner (:839-859)
        rr, rc, rv = rows[~is_local], cols[~is_local], vals[~is_local]
        order = np.lexsort((rr, rc))
        rr, rc, rv = rr[order], rc[order], rv[order]
        if len(rc):
            new_col = np.concatenate(([True], rc[1:] != rc[:-1]))
            distinct = rc[new_col]
            starts = np.flatnonzero(new_col)
            nnzPerCol_remote = np.diff(np.concatenate((starts, [len(rc)]))).astype(I32)
        else:
            distinct = np.zeros(0, I64)
            nnzPerCol_remote = np.zeros(0, I32)
        owner_of_distinct = np.searchsorted(col_split, distinct, side="right") - 1
        owner_of_entry = np.searchsorted(col_split, rc, side="right") - 1
        recvCount = np.bincount(owner_of_distinct, minlength=nprocs).astype(I32) if len(distinct) else np.zeros(nprocs, I32)
        nnzPerProc = np.bincount(owner_of_entry, minlength=nprocs).astype(I64) if len(rc) else np.zeros(nprocs, I64)
        nnzPerProcScan = np.concatenate(([0], np.cumsum(nnzPerProc))).astype(I64)
        rdispls = np.concatenate(([0], np.cumsum(recvCount)[:-1])).astype(I32)
        for owner in range(nprocs):
            requested[r][owner] = distinct[owner_of_distinct == owner]
        per_rank.append(dict(M=M, r0=r0, c0=c0, c1=c1, nnzPerRow_local=nnzPerRow_local, col_local=col_local,
                             val_local=val_local, row_remote=rr.astype(I32), val_remote=rv,
                             nnzPerCol_remote=nnzPerCol_remote, nnzPerProcScan=nnzPerProcScan,
                             recvCount=recvCount, rdispls=rdispls))
    for r in range(nprocs):
        d = per_rank[r]
        # sendCount[dst] = recvCount of dst for owner r (the MPI_Alltoall at :908-909)
        sendCount = np.array([len(requested[dst][r]) for dst in range(nprocs)], I32)
        vdispls = np.concatenate(([0], np.cumsum(sendCount)[:-1])).astype(I32)
        vIndex = (np.concatenate([requested[dst][r] for dst in range(nprocs)]) - d["c0"]).astype(I32) \
            if sendCount.sum() else np.zeros(0, I32)
        recvCount = d["recvCount"]
        ops.append(Operator(
            kind=kind, level=level, M=d["M"], Mbig=n_rows, Nbig=n_cols, row_offset=d["r0"], col_offset=d["c0"],
            n_local_cols=d["c1"] - d["c0"], nnzPerRow_local=d["nnzPerRow_local"], col_local=d["col_local"],
            val_local=d["val_local"], row_remote=d["row_remote"], val_remote=d["val_remote"],
            nnzPerCol_remote=d["nnzPerCol_remote"], nnzPerProcScan=d["nnzPerProcScan"], vIndex=vIndex,
            vdispls=vdispls, rdispls=d["rdispls"],
            sendProcRank=_i32(np.flatnonzero(sendCount)), sendProcCount=_i32(sendCount[sendCount != 0]),
            recvProcRank=_i32(np.flatnonzero(recvCount)), recvProcCount=_i32(recvCount[recvCount != 0]),
            use_double=use_double, nprocs=nprocs, rank=r))
    return ops


def operator_to_global_csr(op: Operator):
    """Inverse of split_operator for a one-rank operator: (indptr, indices, data) with global ids."""
    assert op.nprocs == 1 and op.nnz_remote == 0
    return csr_from_counts(op.nnzPerRow_local), op.col_local.astype(I32), op.val_local


def split_imbalance(indptr: np.ndarray, split: Sequence[int]) -> float:
    """max over ranks of a block's nnz / the mean block nnz"""
    split = np.asarray(split, I64)
    per = np.asarray(indptr, I64)[split[1:]] - np.asarray(indptr, I64)[split[:-1]]
    return float(per.max() * len(per) / max(int(per.sum()), 1))


def partition_hierarchy(h: Hierarchy, nprocs: int, agglomerate_below: int = 0,
                        align_coarse: bool = True, rebalance_above: float = 0.0) -> List[Hierarchy]:
    """Row-partition a one-rank hierarchy over `nprocs` ranks, keeping Saena's layout per rank.

    Level 0 uses nnz-balanced contiguous row blocks; each coarse level follows the level above
    (`aligned_coarse_split`: an aggregate lives where its root lives), so a level's vectors never
    change partition between R's output and the coarse grid
    (Ac.split_old == Ac.split: Grid::repart_u is the identity) -- except below
    `agglomerate_below` global rows, where the level and everything coarser lives on rank 0 and
    the repart plan gathers/scatters the coarse vector (the reference's shrink-to-one-rank case,
    /root/reference/src/saena_matrix_shrink.cpp:67-96).  The coarsest level is always on rank 0
    (decide_shrinking_c, same file), where the direct solve runs.

    `rebalance_above` > 0: a coarse level whose aligned partition leaves one rank with more than
    that multiple of the mean nnz is split by its own nnz balance instead -- the monotone aligned
    rule drifts (256^3 Poisson on 8 ranks: rank 0 keeps 16 % of the mean at level 4, the last rank
    three times the mean), and the heaviest rank sets the time of every operator application.
    R and P are then simply partitioned by that split too (what the reference's `repart` achieves
    by moving Ac after the fact, /root/reference/src/saena_matrix_repart.cpp:728-979); the levels
    below follow the re-balanced one.  Grid::repart_u stays the identity.

    `align_coarse=False` splits every coarse level by its own nnz balance instead (what the
    reference's `repart` may do after coarsening): coarse and fine blocks then do not line up, the
    transfer operators get fat remote parts and whole rows without a single local entry -- kept
    as a stress case for the tests.
    """
    assert h.nprocs == 1
    L = len(h.levels)
    splits = []
    agglomerated = []
    aligned = []   # partition R of level l-1 writes into: follows level l-1's rows
    for l, lv in enumerate(h.levels):
        indptr = csr_from_counts(lv.A.nnzPerRow_local)
        agg = l > 0 and (lv.A.Mbig < agglomerate_below or agglomerated[-1] or l == L - 1)
        agglomerated.append(bool(agg))
        if l == 0:
            aligned.append(None)
            sp = balanced_split(indptr, nprocs)
        else:
            Rp = h.levels[l - 1].R
            if agglomerated[l - 1]:
                al = np.concatenate(([0], np.full(nprocs, lv.A.Mbig))).astype(I64)
            elif not align_coarse:
                al = np.asarray(balanced_split(indptr, nprocs), I64)
            else:
                al = aligned_coarse_split(csr_from_counts(Rp.nnzPerRow_local), Rp.col_local, Rp.val_local,
                                          splits[l - 1])
                if rebalance_above > 0 and not agg and split_imbalance(indptr, al) > rebalance_above:
                    al = np.asarray(balanced_split(indptr, nprocs), I64)
            aligned.append(al)
            sp = np.concatenate(([0], np.full(nprocs, lv.A.Mbig))).astype(I64) if agg else al
        splits.append(np.asarray(sp, I64))
    # the partition R writes into (split_old of level l+1): balanced unless level l itself is agglomerated
    out = [Hierarchy(levels=[], coarse_n=h.coarse_n, coarse_row=h.coarse_row, coarse_col=h.coarse_col,
                     coarse_val=h.coarse_val, nprocs=nprocs, rank=r, scale=h.scale) for r in range(nprocs)]
    for l, lv in enumerate(h.levels):
        ip, ix, dv = operator_to_global_csr(lv.A)
        A_parts = split_operator(KIND_A, l, ip, ix, dv, lv.A.Nbig, splits[l], splits[l], lv.A.use_double)
        for part in A_parts:
            part.use_dense = lv.A.use_dense
        P_parts = R_parts = None
        split_old_next = None
        if lv.P is not None:
            # R produces the coarse vector in the aligned partition; it differs from the coarse
            # grid's own partition only where that grid is agglomerated onto rank 0
            split_old_next = aligned[l + 1]
            ip, ix, dv = operator_to_global_csr(lv.P)
            P_parts = split_operator(KIND_P, l, ip, ix, dv, lv.P.Nbig, splits[l], split_old_next, lv.P.use_double)
            ip, ix, dv = operator_to_global_csr(lv.R)
            R_parts = split_operator(KIND_R, l, ip, ix, dv, lv.R.Nbig, split_old_next, splits[l], lv.R.use_double)
        for r in range(nprocs):
            r0, r1 = int(splits[l][r]), int(splits[l][r + 1])
            level = Level(level=l, A=A_parts[r], inv_diag=lv.inv_diag[r0:r1].copy(), eig_max=lv.eig_max,
                          P=P_parts[r] if P_parts else None, R=R_parts[r] if R_parts else None,
                          active=(r1 > r0),
                          inv_sq_diag=None if lv.inv_sq_diag is None else lv.inv_sq_diag[r0:r1].copy())
            if lv.P is not None:
                so, sn = split_old_next, splits[l + 1]
                level.M_coarse_old = int(so[r + 1] - so[r])
                level.M_coarse = int(sn[r + 1] - sn[r])
                level.repart_send, level.repart_recv = repart_plan(so, sn, r)
            out[r].levels.append(level)
    return out


def repart_plan(so: Sequence[int], sn: Sequence[int], rank: int):
    """Grid::repart_u's plan for `rank`, moving the coarse vector from partition `so` (where R writes it) to `sn`
    (where the coarse grid lives): the overlap of my old block with every new block, (peer, offset_in_old, count)
    to send, and of my new block with every old block, (peer, offset_in_new, count) to receive.  Empty when so == sn."""
    send, recv = [], []
    if not np.array_equal(so, sn):
        for peer in range(len(so) - 1):
            a, b = max(so[rank], sn[peer]), min(so[rank + 1], sn[peer + 1])
            if b > a:
                send.append((peer, int(a - so[rank]), int(b - a)))
            a, b = max(sn[rank], so[peer]), min(sn[rank + 1], so[peer + 1])
            if b > a:
                recv.append((peer, int(a - sn[rank]), int(b - a)))
    return send, recv


def coarse_placement(nprocs: int, n_rows: int, coarsest: bool, above_on_0: bool, agglomerate_below: int,
                     rebalance_above: float, aligned: Sequence[int], imbalance, balanced):
    """Where coarse level l+1 of the torch-built hierarchies lives -- partition_hierarchy's rules, for builders that
    know the level only through the arguments: `n_rows` its global rows, `aligned` the split that follows level l's
    rows, `imbalance()` the level's split_imbalance under `aligned`, `balanced()` its nnz-balanced split.
    `above_on_0`: level l lives on rank 0 alone.  Returns (the split R of level l writes into, the level's own split,
    agglomerated onto rank 0?)."""
    all_on_0 = np.concatenate(([0], np.full(nprocs, n_rows))).astype(I64)
    agg = nprocs > 1 and (n_rows < agglomerate_below or above_on_0 or coarsest)
    al = all_on_0 if above_on_0 else np.asarray(aligned, I64)
    if rebalance_above > 0 and not agg and imbalance() > rebalance_above:
        al = np.asarray(balanced(), I64)
    return al, (all_on_0 if agg else al), agg


# --------------------------------------------------------------------------------------
# (de)serialisation: a flat dict of numpy arrays (np.savez friendly) -- used for the golden
# fixtures under tests/golden/ and for handing a hierarchy between processes.
# --------------------------------------------------------------------------------------
_OP_ARRAYS = ("nnzPerRow_local", "col_local", "val_local", "row_remote", "val_remote", "nnzPerCol_remote",
              "nnzPerProcScan", "vIndex", "vdispls", "rdispls", "sendProcRank", "sendProcCount", "recvProcRank",
              "recvProcCount")
_OP_SCALARS = ("kind", "level", "M", "Mbig", "Nbig", "row_offset", "col_offset", "n_local_cols", "use_double",
               "nprocs", "rank", "use_dense")   # fixtures written before use_dense existed hold 11 values: zip stops there


def hierarchy_to_arrays(h: Hierarchy) -> dict:
    out = {"meta": np.array([len(h.levels), h.coarse_n, h.nprocs, h.rank, int(h.scale)], I64),
           "coarse_row": h.coarse_row, "coarse_col": h.coarse_col, "coarse_val": h.coarse_val}
    for lv in h.levels:
        p = f"L{lv.level}."
        out[p + "inv_diag"] = lv.inv_diag
        if lv.inv_sq_diag is not None:
            out[p + "inv_sq_diag"] = lv.inv_sq_diag
        out[p + "scalars"] = np.array([lv.eig_max, float(lv.active), lv.M_coarse_old, lv.M_coarse,
                                       float(lv.P is not None)], F64)
        out[p + "repart_send"] = np.array(lv.repart_send, I32).reshape(-1, 3)
        out[p + "repart_recv"] = np.array(lv.repart_recv, I32).reshape(-1, 3)
        for name, op in (("A", lv.A), ("P", lv.P), ("R", lv.R)):
            if op is None:
                continue
            q = p + name + "."
            out[q + "scalars"] = np.array([int(getattr(op, s)) for s in _OP_SCALARS], I64)
            for a in _OP_ARRAYS:
                out[q + a] = getattr(op, a)
    return out


def hierarchy_from_arrays(d) -> Hierarchy:
    meta = [int(x) for x in d["meta"]]
    nlev, coarse_n, nprocs, rank = meta[:4]
    scale = bool(meta[4]) if len(meta) > 4 else False
    keys = set(d.files) if hasattr(d, "files") else set(d.keys())
    levels = []
    for l in range(nlev):
        p = f"L{l}."
        eig, active, mco, mc, has_p = d[p + "scalars"]

        def op(name):
            q = p + name + "."
            sc = dict(zip(_OP_SCALARS, (int(x) for x in d[q + "scalars"])))
            sc["use_double"] = bool(sc["use_double"])
            sc["use_dense"] = bool(sc.get("use_dense", 0))
            return Operator(**sc, **{a: np.array(d[q + a]) for a in _OP_ARRAYS})

        lv = Level(level=l, A=op("A"), inv_diag=np.array(d[p + "inv_diag"]), eig_max=float(eig), active=bool(active),
                   M_coarse_old=int(mco), M_coarse=int(mc),
                   repart_send=[tuple(int(x) for x in r) for r in d[p + "repart_send"]],
                   repart_recv=[tuple(int(x) for x in r) for r in d[p + "repart_recv"]],
                   inv_sq_diag=np.array(d[p + "inv_sq_diag"]) if (p + "inv_sq_diag") in keys else None)
        if has_p:
            lv.P, lv.R = op("P"), op("R")
        levels.append(lv)
    return Hierarchy(levels=levels, coarse_n=coarse_n, coarse_row=np.array(d["coarse_row"]),
                     coarse_col=np.array(d["coarse_col"]), coarse_val=np.array(d["coarse_val"]), nprocs=nprocs,
                     rank=rank, scale=scale)
