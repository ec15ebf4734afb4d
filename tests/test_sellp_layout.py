"""Mapping 101 (sliced layout over rows sorted by length inside 256-row windows), the half that needs no GPU:
saena_b200_sellp_layout -- the function the device build calls -- gives the permutation and the slice offsets; the
fill kernel and the product kernel (csrc/operator.cu:sliced_fill_kernel, csrc/spmv_kernels.cuh:spmv_sellp_body) are
restated in numpy on top of it, index for index, and must reproduce the CSR product.  The kernels themselves are
tested on the GPU (tests/test_zz_dense_levels_gpu.py::test_sorted_sliced_layout_mapping_101)."""
import numpy as np
import pytest

from saena_b200.native import sellp_layout
from tests.util import GOLDEN_EXTRA, Golden


def _emulate(rowptr, col, val, x):
    """sliced_fill_kernel + spmv_sellp_body, slot by slot"""
    M = len(rowptr) - 1
    perm, sp = sellp_layout(rowptr)
    n_slots = len(perm)
    scol = np.zeros(max(int(sp[-1]), 1), np.int64)
    sval = np.zeros(max(int(sp[-1]), 1))
    for slot in range(n_slots):                       # sliced_fill_kernel
        sl, lane = slot >> 5, slot & 31
        base, ln = int(sp[sl]), int(sp[sl + 1] - sp[sl]) >> 5
        row = int(perm[slot])
        a, b = (int(rowptr[row]), int(rowptr[row + 1])) if row >= 0 else (0, 0)
        pad_col = int(col[b - 1]) if b > a else 0
        for j in range(ln):
            dst = base + j * 32 + lane
            scol[dst], sval[dst] = (col[a + j], val[a + j]) if a + j < b else (pad_col, 0.0)
    y = np.full(M, np.nan)
    for vb in range(n_slots // 256):                  # spmv_sellp_body, one CTA per window
        s_sum = np.full(256, np.nan)
        for t in range(256):
            slot = vb * 256 + t
            sl, lane = slot >> 5, t & 31
            base, ln = int(sp[sl]), int(sp[sl + 1] - sp[sl]) >> 5
            s = 0.0
            for j in range(ln):
                s += sval[base + j * 32 + lane] * x[scol[base + j * 32 + lane]]
            if perm[slot] >= 0:
                s_sum[perm[slot] - vb * 256] = s      # back to row order through shared memory
        for t in range(256):
            if vb * 256 + t < M:
                y[vb * 256 + t] = s_sum[t]
    return y, perm, sp


def _csr(op):
    rp = np.zeros(op.M + 1, np.int64)
    np.cumsum(op.nnzPerRow_local, out=rp[1:])
    return rp, op.col_local.astype(np.int64) - op.col_offset, op.val_local


@pytest.mark.parametrize("M,seed", [(0, 0), (1, 1), (31, 2), (256, 3), (257, 4), (700, 5)])
def test_layout_on_random_ragged_rows(M, seed):
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 40, M) * (rng.uniform(size=M) > 0.1)           # some empty rows
    rp = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    ncols = 97
    col = rng.integers(0, ncols, int(rp[-1]))
    val = rng.uniform(-1, 1, int(rp[-1]))
    x = rng.uniform(-1, 1, ncols)
    y, perm, sp = _emulate(rp, col, val, x)
    want = np.array([np.dot(val[rp[i]:rp[i + 1]], x[col[rp[i]:rp[i + 1]]]) for i in range(M)])
    assert np.allclose(y, want, rtol=1e-13, atol=1e-15)
    # a permutation of the rows of each window, sorted by length, longest first, ties in row order
    n_slots = (M + 255) // 256 * 256
    assert len(perm) == n_slots and len(sp) == n_slots // 32 + 1
    for w in range(n_slots // 256):
        p = perm[w * 256:(w + 1) * 256]
        rows = p[p >= 0]
        assert sorted(rows.tolist()) == list(range(w * 256, min(M, (w + 1) * 256))) and np.all(p[len(rows):] == -1)
        ln = lens[rows]
        assert np.all(np.diff(ln) <= 0)
        assert all(rows[k] < rows[k + 1] for k in range(len(rows) - 1) if ln[k] == ln[k + 1])
    # padding: never more than the unsorted sliced layout's
    pad_sorted = int(sp[-1])
    padded = np.zeros((M + 31) // 32 * 32, np.int64)
    padded[:M] = lens
    assert pad_sorted <= int(padded.reshape(-1, 32).max(axis=1).sum()) * 32 if M else pad_sorted == 0


def test_layout_on_the_irregular_golden_operators():
    g = Golden(GOLDEN_EXTRA[0])       # Helmholtz2D: 24..40 entries per row
    rng = np.random.default_rng(9)
    for lv in g.hier.levels:
        for op in (lv.A, lv.P, lv.R):
            if op is None:
                continue
            rp, col, val = _csr(op)
            x = rng.uniform(-1, 1, op.n_local_cols)
            y, _, sp = _emulate(rp, col, val, x)
            assert np.allclose(y, op.to_scipy_local() @ x, rtol=1e-13, atol=1e-14)
            assert int(sp[-1]) >= op.nnz_local
