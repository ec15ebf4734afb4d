"""Mapping 103 (symmetric diagonals), the half that needs no GPU: the host rule through the C ABI
(saena_b200_symdiag_plan), and the fill, the symmetry check and the kernel's sum order restated in numpy
(tests/symdiag_cases.py), which must reproduce the CSR row sums bit for bit.  The kernels themselves are tested on the
GPU (tests/test_zz_symdiag_gpu.py)."""
import numpy as np
import pytest

from saena_b200.native import symdiag_plan
from tests import symdiag_cases as sc
from tests.util import Golden


def _eligible_cases():
    yield "7pt_37x23x19", sc.stencil((37, 23, 19), 0, seed=1)
    yield "27pt_13x11x9", sc.stencil((13, 11, 9), 1, seed=2)
    yield "band8_1500", sc.band(1500, 8)
    yield "band5_1500", sc.band(1500, 5)


@pytest.mark.parametrize("name,csr", list(_eligible_cases()), ids=lambda v: v if isinstance(v, str) else "")
def test_symdiag_sums_are_the_csr_sums(name, csr):
    rp, col, val = csr
    stored = sc.plan(rp, col)
    assert stored is not None, name
    want_nd = {"7pt_37x23x19": 4, "27pt_13x11x9": 14, "band8_1500": 9, "band5_1500": 6}[name]
    assert len(stored) == want_nd and stored[0] == 0 and stored == sorted(stored)
    d = sc.fill_and_check(rp, col, val, stored)
    assert d is not None
    assert np.count_nonzero(d) == np.count_nonzero(val[col >= sc.rows_of(rp)])   # every upper entry, once
    rng = np.random.default_rng(3)
    for x in (rng.uniform(-1, 1, len(rp) - 1), np.ones(len(rp) - 1)):
        assert sc.bitwise_equal_sums(sc.symdiag_sums(d, stored, x), sc.csr_sums(rp, col, val, x)), name


def test_bench_level0_operator_is_eligible():
    """the 7-point Poisson operator as the setup uploads it (sorted columns, exactly symmetric values)"""
    from saena_b200 import sa_setup
    h = sa_setup.build_device_hierarchy(*sa_setup.poisson3d_coo(12), device="cpu").to_rank(0, 1)
    rp, col, val = sc.csr_of(h.levels[0].A)
    stored = sc.plan(rp, col)
    assert stored == [0, 1, 12, 144]
    assert sc.fill_and_check(rp, col, val, stored) is not None


def test_refused_for_an_unstructured_matrix():
    rp, col, _ = sc.csr_of(Golden("helmholtz2d_p8").hier.levels[0].A)
    assert sc.plan(rp, col) is None


def test_refused_for_a_non_symmetric_stencil():
    rp, col, val = sc.stencil((9, 8, 7), 0, seed=4, upwind=0.25)   # symmetric pattern, values not
    stored = sc.plan(rp, col)
    assert stored == [0, 1, 9, 72]
    assert sc.fill_and_check(rp, col, val, stored) is None
    up = col >= sc.rows_of(rp)                                     # one-sided pattern: no mirror offsets
    one_sided_rp = np.concatenate(([0], np.cumsum(np.bincount(sc.rows_of(rp)[up], minlength=len(rp) - 1))))
    assert sc.plan(one_sided_rp, col[up]) is None


def test_refused_for_the_band_golden_operator():
    """band8_1500 as the reference stored it: the pattern of sc.band(1500, 8), but a_ij and a_ji differ in the last
    bits for some pairs"""
    rp, col, val = sc.csr_of(Golden("band8_1500").hier.levels[0].A)
    stored = sc.plan(rp, col)
    assert stored == list(range(9))
    assert sc.fill_and_check(rp, col, val, stored) is None


def test_refused_for_a_row_whose_columns_do_not_ascend():
    rp, col, val = sc.stencil((9, 8, 7), 0, seed=5)
    stored = sc.plan(rp, col)
    r = 100
    col, val = col.copy(), val.copy()
    col[[rp[r], rp[r] + 1]] = col[[rp[r] + 1, rp[r]]]
    val[[rp[r], rp[r] + 1]] = val[[rp[r] + 1, rp[r]]]
    assert sc.plan(rp, col) == stored                 # the same offsets: only the device's order check refuses it
    assert sc.fill_and_check(rp, col, val, stored) is None


def test_refused_for_one_value_changed_by_one_ulp():
    rp, col, val = sc.stencil((9, 8, 7), 0, seed=5)
    stored = sc.plan(rp, col)
    assert sc.fill_and_check(rp, col, val, stored) is not None
    for lower in (True, False):
        k = int(np.flatnonzero((col < sc.rows_of(rp)) if lower else (col > sc.rows_of(rp)))[17])
        v = val.copy()
        v[k] = np.nextafter(v[k], np.inf)
        assert sc.fill_and_check(rp, col, v, stored) is None


def test_refused_for_more_than_32_offsets():
    M, nnz = 100000, 3300000
    for half, want in ((15, 16), (16, None)):        # 31 offsets: 16 stored; 33 offsets: refused
        off = np.arange(-half, half + 1, dtype=np.int32)
        got = symdiag_plan(M, off, nnz, nnz)
        assert (got is None) if want is None else (len(got) == want and got == list(range(16)))
    # 16 mirrored pairs without offset 0 are 32 offsets but 17 stored diagonals: more than the kernel holds
    off = np.concatenate((-np.arange(1, 17), np.arange(1, 17))).astype(np.int32)
    assert symdiag_plan(M, off, nnz, nnz) is None


def test_refused_where_it_streams_no_fewer_bytes():
    M = 10000
    off = np.array([-5000, -1, 0, 1, 5000], np.int32)
    assert symdiag_plan(M, off, 5 * M, 5 * M) == [0, 1, 5000]       # 24 B/row against 0.75 * 60
    assert symdiag_plan(M, off, 2 * M + 10, 2 * M + 10) is None      # the off-diagonals nearly empty
    assert symdiag_plan(M, off[1:4], 3 * M, 3 * M) == [0, 1]
    assert symdiag_plan(M, np.array([-1, 0], np.int32), 2 * M, 2 * M) is None   # no mirror of -1
    assert symdiag_plan(0, np.zeros(0, np.int32), 0, 0) is None
