"""Mapping 103 (symmetric diagonals, csrc/spmv_kernels.cuh:spmv_symdiag_kernel) on the GPU.  Forced on the operators
of tests/symdiag_cases.py it must give the sliced layout's results (mapping 100) bit for bit -- matvec, residual, the
Chebyshev and Jacobi sweeps -- and match scipy; operators that are not eligible keep the rule's mapping; a value update
keeps the layout when the new values are symmetric and moves the operator to the sliced layout when they are not; and a
PCG solve on the 64^3 bench hierarchy gives the same bits whichever layout level 0 runs on."""
import numpy as np
import pytest

from tests import symdiag_cases as sc
from tests.util import Golden, rel


def _cuda() -> bool:
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _cuda(), reason="needs a CUDA device")]

SELL, SELLP, SYMDIAG = 100, 101, 103
CASES = {"7pt_37x23x19": lambda: sc.stencil((37, 23, 19), 0, seed=1),
         "27pt_13x11x9": lambda: sc.stencil((13, 11, 9), 1, seed=2),
         "band8_1500": lambda: sc.band(1500, 8),    # 9 stored diagonals: the 16-diagonal kernel
         "band5_1500": lambda: sc.band(1500, 5)}    # 6: the 8-diagonal kernel


def _one_level(rp, col, val):
    """a lone level-0 operator (matvec / residual / smooth hooks)"""
    from saena_b200.hierarchy import F64, I32, KIND_A, Hierarchy, Level, Operator
    M = len(rp) - 1
    op = Operator(kind=KIND_A, level=0, M=M, Mbig=M, Nbig=M, row_offset=0, col_offset=0, n_local_cols=M,
                  nnzPerRow_local=np.diff(rp).astype(I32), col_local=col.astype(I32), val_local=val.astype(F64))
    diag = np.array([val[rp[i]:rp[i + 1]][col[rp[i]:rp[i + 1]] == i].sum() for i in range(M)])
    return Hierarchy([Level(0, op, inv_diag=1.0 / diag, eig_max=1.9)], coarse_n=0)


def _context(rp, col, val, mapping):
    from saena_b200.native import Context
    ctx = Context()
    ctx.upload_hierarchy(_one_level(rp, col, val))
    ctx.set_mapping(0, 0, mapping)
    return ctx


def _outputs(ctx, M):
    rng = np.random.default_rng(11)
    x, rhs = rng.uniform(-1, 1, M), rng.uniform(-1, 1, M)
    return {"matvec": ctx.matvec(0, 0, x), "residual": ctx.residual(0, x, rhs),
            "chebyshev": ctx.smooth(0, "chebyshev", 3, x, rhs), "jacobi": ctx.smooth(0, "jacobi", 2, x, rhs),
            "chebyshev_from_zero": ctx.smooth(0, "chebyshev", 2, np.zeros(M), rhs)}


@pytest.mark.parametrize("name", list(CASES))
def test_forced_symdiag_gives_the_sliced_bits(name):
    rp, col, val = CASES[name]()
    M = len(rp) - 1
    ctx = _context(rp, col, val, SELL)
    try:
        assert ctx.get_mapping(0, 0) == SELL
        want = _outputs(ctx, M)
        sell_bytes = ctx.operator_bytes(0, 0)
        ctx.set_mapping(0, 0, SYMDIAG)
        assert ctx.get_mapping(0, 0) == SYMDIAG
        got = _outputs(ctx, M)
        nd = len(sc.plan(rp, col))
        assert ctx.operator_bytes(0, 0) == 8 * nd * M + 16 * M < sell_bytes
        for k in want:
            assert sc.bitwise_equal_sums(got[k], want[k]), (name, k)
        import scipy.sparse as sp
        x = np.random.default_rng(11).uniform(-1, 1, M)
        assert rel(got["matvec"], sp.csr_matrix((val, col, rp), shape=(M, M)) @ x) <= 1e-13
        ctx.set_mapping(0, 0, SELLP)
        assert all(np.array_equal(_outputs(ctx, M)[k], want[k]) for k in want)
    finally:
        ctx.close()


def test_ineligible_operators_keep_the_rule():
    from saena_b200.native import Context
    rp, col, val = sc.stencil((9, 8, 7), 0, seed=5)
    off_by_ulp = val.copy()
    off_by_ulp[int(np.flatnonzero(col < sc.rows_of(rp))[17])] *= 1.0 + 2.0 ** -52   # one lower value, one ulp up
    unsorted_col, unsorted_val = col.copy(), val.copy()                      # the same matrix, one row's first two
    r = 100                                                                   # entries stored in descending order
    unsorted_col[[rp[r], rp[r] + 1]] = col[[rp[r] + 1, rp[r]]]
    unsorted_val[[rp[r], rp[r] + 1]] = val[[rp[r] + 1, rp[r]]]
    cases = [sc.stencil((9, 8, 7), 0, seed=4, upwind=0.25),                 # symmetric pattern, values not
             (rp, col, off_by_ulp),
             (rp, unsorted_col, unsorted_val),
             sc.csr_of(Golden("band8_1500").hier.levels[0].A)]              # a_ij, a_ji differ in the last bits
    for case in cases:
        ctx = _context(*case, 0)
        try:
            rule = ctx.get_mapping(0, 0)
            ctx.set_mapping(0, 0, SYMDIAG)
            assert ctx.get_mapping(0, 0) == rule
        finally:
            ctx.close()
    g = Golden("helmholtz2d_p8")                                             # unstructured
    ctx = Context()
    try:
        ctx.upload_hierarchy(g.hier)
        for l in range(len(g.hier.levels)):
            rule = ctx.get_mapping(l, 0)
            ctx.set_mapping(l, 0, SYMDIAG)
            assert ctx.get_mapping(l, 0) == rule, l
    finally:
        ctx.close()


def test_value_updates():
    rp, col, val = CASES["7pt_37x23x19"]()
    M = len(rp) - 1
    x = np.random.default_rng(5).uniform(-1, 1, M)
    sym = sc.stencil((37, 23, 19), 0, seed=7)[2]                             # new symmetric values
    asym = sc.stencil((37, 23, 19), 0, seed=7, upwind=0.5)[2]                # same pattern, not symmetric
    ctx = _context(rp, col, val, SYMDIAG)
    try:
        assert ctx.get_mapping(0, 0) == SYMDIAG
        ctx.update_values(sym)
        assert ctx.get_mapping(0, 0) == SYMDIAG
        fresh = _context(rp, col, sym, SYMDIAG)
        try:
            assert np.array_equal(ctx.matvec(0, 0, x), fresh.matvec(0, 0, x))
        finally:
            fresh.close()
        ctx.update_values(asym)
        assert ctx.get_mapping(0, 0) == SELL
        fresh = _context(rp, col, asym, SELL)
        try:
            assert np.array_equal(ctx.matvec(0, 0, x), fresh.matvec(0, 0, x))
        finally:
            fresh.close()
        ctx.update_values(sym)                                                # symmetric again: eligible again
        ctx.set_mapping(0, 0, SYMDIAG)
        assert ctx.get_mapping(0, 0) == SYMDIAG
        fresh = _context(rp, col, sym, SELL)
        try:
            assert sc.bitwise_equal_sums(ctx.matvec(0, 0, x), fresh.matvec(0, 0, x))
        finally:
            fresh.close()
    finally:
        ctx.close()


def test_pcg_on_the_bench_hierarchy_is_the_same_on_every_level0_layout():
    import torch
    from saena_b200 import sa_setup
    from saena_b200.native import Context
    n = 64
    dh = sa_setup.build_device_hierarchy(*sa_setup.poisson3d_coo(n), device="cuda")
    h = dh.to_rank(0, 1)
    del dh
    torch.cuda.empty_cache()
    rhs = sa_setup.poisson3d_rhs(n)
    ctx = Context()
    try:
        ctx.upload_hierarchy(h)
        assert ctx.get_mapping(0, 0) == SYMDIAG          # 262 144 rows: the rule's choice for an eligible operator
        runs = {}
        for m in (SELL, SELLP, SYMDIAG):
            ctx.set_mapping(0, 0, m)
            assert ctx.get_mapping(0, 0) == m
            runs[m] = ctx.solve_pcg(rhs)
        u, iters, hist = runs[SELL]
        assert iters > 0
        for m in (SELLP, SYMDIAG):
            assert runs[m][1] == iters, m
            assert np.array_equal(runs[m][2], hist), m
            assert np.array_equal(runs[m][0], u), m
    finally:
        ctx.close()
