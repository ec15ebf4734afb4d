"""Host reference of saena_b200_update_values (no device): the hierarchy the update should leave behind, with scipy.

A_0 takes the new values; A_{l+1} = R_l A_l P_l mapped onto the stored pattern of A_{l+1} by the setup's filter rule
(sa_setup_dist.filter_entries_dist): a stored entry takes the product's value, an off-diagonal entry outside the pattern
is lumped into its row's diagonal, a diagonal below ALMOST_ZERO in magnitude (or one the product lacks) is 1; a stored
off-diagonal the product lacks is an error.  One-rank hierarchies only (local column ids are global ones)."""
import copy

import numpy as np
import scipy.sparse as sp

from saena_b200.sa_setup import ALMOST_ZERO


def _csr(op, val=None):
    indptr = np.zeros(op.M + 1, np.int64)
    np.cumsum(op.nnzPerRow_local, out=indptr[1:])
    return sp.csr_matrix((op.val_local if val is None else val, op.col_local - op.col_offset, indptr),
                         shape=(op.M, op.n_local_cols))


def map_onto_pattern(C: sp.csr_matrix, op):
    """(values of op's stored pattern in stored order, lumped fraction) for the product C"""
    C = C.tocsr()
    C.sort_indices()
    n = op.M
    indptr = np.zeros(n + 1, np.int64)
    np.cumsum(op.nnzPerRow_local, out=indptr[1:])
    scol = np.asarray(op.col_local, np.int64) - op.col_offset
    srow = np.repeat(np.arange(n), np.diff(indptr))
    crow = np.repeat(np.arange(n), np.diff(C.indptr))
    ccol, cval = C.indices.astype(np.int64), C.data
    skey, ckey = srow * n + scol, crow * n + ccol
    order = np.argsort(skey, kind="stable")
    pos = np.searchsorted(skey[order], ckey)
    pos = np.minimum(pos, len(skey) - 1)
    found = skey[order][pos] == ckey
    c_diag = crow == ccol
    val = np.zeros(len(skey))
    val[order[pos[found]]] = cval[found]
    have = np.zeros(len(skey), bool)
    have[order[pos[found]]] = True
    if np.any((srow != scol) & ~have):
        raise ValueError("A_{l+1} is not a Galerkin product of the level above")
    lumped = ~found & ~c_diag
    lump = np.bincount(crow[lumped], weights=cval[lumped], minlength=n)
    has_cdiag = np.zeros(n, bool)
    has_cdiag[crow[c_diag]] = True
    dpos = np.flatnonzero(srow == scol)
    drow = srow[dpos]
    d = np.where(has_cdiag[drow], val[dpos] + lump[drow], 1.0)
    d = np.where(np.abs(d) < ALMOST_ZERO, 1.0, d)
    val[dpos] = d
    c_norm = np.linalg.norm(cval)
    frac = float(np.linalg.norm(cval[lumped]) / c_norm) if c_norm > 0 else 0.0
    return val, frac


def updated_hierarchy(h, val0):
    """(hierarchy with the new values, inv_diag and coarsest COO; eig_max left as stored, lumped fractions)"""
    h = copy.deepcopy(h)
    val0 = np.asarray(val0, np.float64)
    h.levels[0].A.val_local = val0.copy()
    fracs = [0.0]
    for l in range(len(h.levels)):
        lv = h.levels[l]
        A = _csr(lv.A)
        lv.inv_diag = 1.0 / A.diagonal()
        if lv.P is None:
            continue
        C = _csr(lv.R) @ (A @ _csr(lv.P))
        nxt = h.levels[l + 1].A
        vals, frac = map_onto_pattern(C, nxt)
        nxt.val_local = vals
        fracs.append(frac)
    last = h.levels[-1].A
    h.coarse_val = np.asarray(last.val_local, np.float64).copy()
    indptr = np.zeros(last.M + 1, np.int64)
    np.cumsum(last.nnzPerRow_local, out=indptr[1:])
    h.coarse_row = np.repeat(np.arange(last.M), np.diff(indptr)).astype(np.int32)
    h.coarse_col = (np.asarray(last.col_local) - last.col_offset).astype(np.int32)
    return h, fracs


def shifted_values(op, sigma):
    """values of A + sigma I in op's stored order (the mass term of an implicit time step)"""
    indptr = np.zeros(op.M + 1, np.int64)
    np.cumsum(op.nnzPerRow_local, out=indptr[1:])
    row = np.repeat(np.arange(op.M), np.diff(indptr))
    return op.val_local + sigma * (row == np.asarray(op.col_local) - op.col_offset)


def rescaled_values(op, dscale):
    """values of D A D, D = diag(dscale), in op's stored order (changes every off-diagonal)"""
    indptr = np.zeros(op.M + 1, np.int64)
    np.cumsum(op.nnzPerRow_local, out=indptr[1:])
    row = np.repeat(np.arange(op.M), np.diff(indptr))
    col = np.asarray(op.col_local, np.int64) - op.col_offset
    return op.val_local * dscale[row] * dscale[col]
