"""Mapping 103 (symmetric diagonals, csrc/operator.cu + csrc/spmv_kernels.cuh:spmv_symdiag_kernel) restated in numpy,
and the operators its tests run on.

- `offsets` / `plan`: the distinct offsets col - row the device pass collects, and the host rule
  (saena_b200_symdiag_plan, called through the C ABI).
- `fill_and_check`: sd_fill_kernel + sd_check_kernel -- upper entries into d_q[row], then every lower entry must be
  present in its mirror row with the same bits, and the lower and upper off-diagonal counts must agree.
- `symdiag_sums`: the kernel's sum order -- lower terms for k descending, d_0[i] x[i], upper terms for k ascending,
  each `sum += a * x` from 0.0, terms outside [0, M) adding 0.0 * 0.0.
- `csr_sums`: the CSR / sliced kernels' order, one row in column order from 0.0.
Both sums multiply, round, then add, as numpy does; the device contracts each step to one fused multiply-add in both
kernels alike.
"""
import numpy as np

from saena_b200.native import symdiag_plan


def csr_of(op):
    """(rowptr int64, local columns int64, values) of an uploaded Operator"""
    rp = np.zeros(op.M + 1, np.int64)
    np.cumsum(op.nnzPerRow_local, out=rp[1:])
    return rp, op.col_local.astype(np.int64) - op.col_offset, np.asarray(op.val_local, np.float64)


def rows_of(rp):
    return np.repeat(np.arange(len(rp) - 1, dtype=np.int64), np.diff(rp))


def offsets(rp, col):
    return np.unique(col - rows_of(rp))


def padded_est(rp):
    """entries of the sliced layout: every 32-row slice padded to its longest row (operator.cu:sliced_padded_est)"""
    lens = np.diff(rp)
    pad = (-len(lens)) % 32
    return int(np.concatenate([lens, np.zeros(pad, np.int64)]).reshape(-1, 32).max(axis=1).sum() * 32)


def plan(rp, col):
    """the stored offsets of the layout, or None where the host rule refuses it"""
    return symdiag_plan(len(rp) - 1, offsets(rp, col).astype(np.int32), int(rp[-1]), padded_est(rp))


def fill_and_check(rp, col, val, stored):
    """d[q, i] = a_{i, i + stored[q]}; None when the values or the pattern are not exactly symmetric or a row's
    columns do not strictly ascend"""
    M = len(rp) - 1
    rows = rows_of(rp)
    if np.any((np.diff(col) <= 0) & (rows[1:] == rows[:-1])):
        return None
    index = {k: q for q, k in enumerate(stored)}
    d = np.zeros((len(stored), M))
    up = col >= rows
    if not all(int(k) in index for k in np.unique(col[up] - rows[up])):
        return None
    for r, c, v in zip(rows[up], col[up], val[up]):
        d[index[int(c - r)], r] = v
    entries = {(int(r), int(c)) for r, c in zip(rows, col)}
    balance = 0
    for r, c, v in zip(rows, col, val):
        if c > r:
            balance -= 1
        if c >= r:
            continue
        balance += 1
        q = index.get(int(r - c))
        if q is None or (int(c), int(r)) not in entries or d[q, c].view(np.int64) != v.view(np.int64):
            return None
    return d if balance == 0 else None


def symdiag_sums(d, stored, x):
    M = d.shape[1]
    i = np.arange(M)
    s = np.zeros(M)

    def term(q, j):
        a = np.where((j >= 0) & (j < M), d[q, np.clip(np.minimum(i, j), 0, M - 1)], 0.0)
        return a * np.where((j >= 0) & (j < M), x[np.clip(j, 0, M - 1)], 0.0)

    for q in range(len(stored) - 1, 0, -1):
        s = s + term(q, i - stored[q])      # a_{i,i-k} = d_k[i-k]
    s = s + d[0] * x
    for q in range(1, len(stored)):
        s = s + term(q, i + stored[q])      # a_{i,i+k} = d_k[i]
    return s


def csr_sums(rp, col, val, x):
    y = np.zeros(len(rp) - 1)
    for i in range(len(y)):
        s = 0.0
        for k in range(rp[i], rp[i + 1]):
            s = s + val[k] * x[col[k]]
        y[i] = s
    return y


def bitwise_equal_sums(a, b):
    """same bits, up to the sign of an all-zero row sum"""
    return np.array_equal(a, b) and np.array_equal(a[a != 0].view(np.int64), b[b != 0].view(np.int64))


# ---- operators --------------------------------------------------------------------------------------------------
def _sym_weight(i, j, seed):
    """a symmetric positive weight of the pair {i, j}: the same bits whichever row asks"""
    lo, hi = np.minimum(i, j), np.maximum(i, j)
    h = (lo * 2654435761 + hi * 40503 + seed * 97) % 1000003
    return 0.5 + h / 1000003.0


def stencil(shape, reach, seed=0, upwind=0.0):
    """CSR of a stencil on a grid of `shape` (natural ordering, x fastest): the neighbours within Chebyshev distance
    `reach` (1: 27-point) or, reach = 0, the 7-point stencil.  Off-diagonal a_ij = -w({i, j}) (symmetric, variable);
    upwind != 0 adds upwind * w to the entry towards +x only (not symmetric); diagonal = 1 + sum of |off-diagonals|."""
    nx, ny, nz = shape
    M = nx * ny * nz
    if reach == 0:
        nbrs = [(1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)]
    else:
        r = range(-reach, reach + 1)
        nbrs = [(a, b, c) for c in r for b in r for a in r if (a, b, c) != (0, 0, 0)]
    idx = np.arange(M)
    ix, iy, iz = idx % nx, (idx // nx) % ny, idx // (nx * ny)
    rows, cols, vals = [idx], [idx], [np.zeros(M)]
    for a, b, c in nbrs:
        ok = (ix + a >= 0) & (ix + a < nx) & (iy + b >= 0) & (iy + b < ny) & (iz + c >= 0) & (iz + c < nz)
        i = idx[ok]
        j = i + a + b * nx + c * nx * ny
        v = -_sym_weight(i, j, seed)
        if upwind and (a, b, c) == (1, 0, 0):
            v = v - upwind * _sym_weight(i, j, seed + 1)
        rows.append(i), cols.append(j), vals.append(v)
    row, col, val = (np.concatenate(t) for t in (rows, cols, vals))
    order = np.lexsort((col, row))
    row, col, val = row[order], col[order], val[order]
    diag = np.zeros(M)
    np.add.at(diag, row, np.abs(val))
    val = np.where(row == col, 1.0 + diag[row], val)
    rp = np.zeros(M + 1, np.int64)
    np.cumsum(np.bincount(row, minlength=M), out=rp[1:])
    return rp, col.astype(np.int64), val


def band(n, b):
    """CSR of saena::band_matrix's pattern and values as the device generates them (operator.cu:band_fill_kernel):
    row i holds columns [i-b, i+b] inside [0, n), value 1/(i+j+1) -- symmetric to the bit"""
    i = np.repeat(np.arange(n, dtype=np.int64), 2 * b + 1)
    j = i + np.tile(np.arange(-b, b + 1, dtype=np.int64), n)
    ok = (j >= 0) & (j < n)
    i, j = i[ok], j[ok]
    rp = np.zeros(n + 1, np.int64)
    np.cumsum(np.bincount(i, minlength=n), out=rp[1:])
    return rp, j, 1.0 / (i + j + 1).astype(np.float64)
