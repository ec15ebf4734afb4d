"""The device SpGEMM of the Galerkin product (csrc/spgemm.cu, SURVEY 8f #3) against an exact reference, and the
hierarchy it builds against the REFERENCE's own coarse operators: the golden files hold A_l, P_l, R_l of every level as
saena_object::setup left them (Ac = R A P through the reference's matmat + MKL product shim), and where oracle/_ref
travelled, the live reference at 32^3.

The products are checked by one checker against tests/spgemm_cases.py's reference: pattern and row offsets exactly,
values bit for bit where the operands make every sum exact, else within the per-entry rounding bound.  The cases
there reach every bin of both passes at and across its edges, hash tables whose probes wrap around, CTAs of the
grid-stride kernels that handle more than one row, thousands of scan blocks, degenerate shapes and entries that cancel
to exactly 0; each case's claim is re-checked against the SM count and shared memory of the card that runs it."""
import numpy as np
import pytest

from tests import spgemm_cases
from tests.util import GOLDEN, Golden

pytestmark = pytest.mark.gpu


def _rand_csr(rng, n_rows, n_cols, row_nnz):
    import scipy.sparse as sp
    counts = np.minimum(np.asarray(row_nnz, np.int64), n_cols)
    indptr = np.concatenate(([0], np.cumsum(counts)))
    cols = np.concatenate([np.sort(rng.choice(n_cols, int(c), replace=False)) for c in counts]) if counts.sum() else np.zeros(0, np.int64)
    vals = rng.uniform(-1, 1, int(counts.sum()))
    return sp.csr_matrix((vals, cols, indptr), shape=(n_rows, n_cols))


def _device_product(A, B):
    import torch
    from saena_b200 import native
    dev = torch.device("cuda")
    t = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a), device=dev).to(dt).contiguous()
    rp, col, val = native.spgemm_csr(A.shape[0], A.shape[1], B.shape[1], t(A.indptr, torch.int64), t(A.indices, torch.int32),
                                     t(A.data, torch.float64), t(B.indptr, torch.int64), t(B.indices, torch.int32),
                                     t(B.data, torch.float64))
    return rp.cpu().numpy(), col.cpu().numpy(), val.cpu().numpy()


def _first(mask, rp):
    i = int(np.argmax(mask))
    return f"first at entry {i} (row {int(np.searchsorted(rp, i, side='right')) - 1})"


def _check_product(A, B):
    """C = A B on the device: row offsets, nnz and columns equal the structural reference, columns strictly ascend in
    each row, a second call gives the same structure bit for bit, and values equal the reference bit for bit where the
    operands make every sum exact (spgemm_cases.values_are_exact), else lie within its per-entry bound"""
    ref = spgemm_cases.reference(A, B)
    rp, col, val = _device_product(A, B)
    bad_rows = np.flatnonzero(np.diff(rp) != np.diff(ref.indptr)) if len(rp) == len(ref.indptr) else []
    assert np.array_equal(rp, ref.indptr), f"row offsets differ: {len(bad_rows)} rows with a wrong count, first {bad_rows[:5]}"
    assert len(col) == len(val) == rp[-1], "nnz differs from rowptr[M]"
    first_of_row = np.zeros(len(col), bool)
    first_of_row[rp[:-1][rp[:-1] < len(col)]] = True
    assert np.all(np.diff(col)[~first_of_row[1:]] > 0), "columns do not strictly ascend inside a row"
    assert np.array_equal(col, ref.indices), "columns differ: " + _first(col != ref.indices, rp)
    rp2, col2, _ = _device_product(A, B)
    assert np.array_equal(rp2, rp) and np.array_equal(col2, col), "a second call gives another structure"
    got = val.astype(np.longdouble)
    if spgemm_cases.values_are_exact(A, B, ref.count):
        wrong = got != ref.value
        assert not wrong.any(), f"{int(wrong.sum())} values differ from the exact reference, " + _first(wrong, rp)
    else:
        wrong = np.abs(got - ref.value) > ref.bound
        assert not wrong.any(), f"{int(wrong.sum())} values outside (k + 1) 2^-53 (|A||B|)_ij, " + _first(wrong, rp)


# (rows of A, inner size, columns of B, nnz per row of A, nnz per row of B): random values in [-1, 1]
CASES = [
    (3000, 2500, 4000, (0, 1, 3, 7), (0, 2, 5)),                  # empty rows, tiny rows: the 32-entry warp tables
    (1200, 900, 5000, (5, 9, 14), (6, 9, 12)),                    # <= 128 / <= 512 entries: the larger warp tables
    (300, 2000, 60000, (40, 60), (50, 70)),                       # ~3000-4000 entries per row: 96 KB CTA tables
    (60, 3000, 200000, (90, 110), (70, 80)),                      # ~7000-8000 entries: 192 KB CTA tables
    (40, 1500, 9000, (400, 500), (300, 400)),                     # nearly dense rows, N <= 24576: dense accumulator in shared memory
    (24, 2500, 90000, (600, 700), (200, 300)),                    # > 8192 entries with N = 90000: dense accumulator slab in global memory
    (16, 40, 40, (40,), (40,)),                                   # dense x dense, N tiny
]


@pytest.mark.parametrize("m,k,n,a_nnz,b_nnz", CASES)
def test_device_spgemm_matches_scipy(m, k, n, a_nnz, b_nnz):
    rng = np.random.default_rng(m + k + n)
    A = _rand_csr(rng, m, k, rng.choice(a_nnz, m))
    B = _rand_csr(rng, k, n, rng.choice(b_nnz, k))
    _check_product(A, B)


@pytest.mark.parametrize("name", spgemm_cases.NAMES)
def test_device_spgemm_at_every_dispatch_edge(name):
    import torch
    case = spgemm_cases.build(name)
    props = torch.cuda.get_device_properties(0)
    unmet = spgemm_cases.unmet_claims(case, props.multi_processor_count, props.shared_memory_per_block_optin)
    assert unmet == [], f"on {props.name} the case does not cover what it claims: {unmet}"
    _check_product(case.A, case.B)


def _same_operator(a, b, tol=1e-13):
    assert (a.M, a.Nbig, a.nnz_local, a.nnz_remote) == (b.M, b.Nbig, b.nnz_local, b.nnz_remote)
    assert np.array_equal(a.nnzPerRow_local, b.nnzPerRow_local)
    assert np.array_equal(a.col_local, b.col_local)
    assert np.max(np.abs(a.val_local - b.val_local)) <= tol * np.max(np.abs(b.val_local))


@pytest.mark.parametrize("name", GOLDEN)
def test_hierarchy_built_with_the_device_spgemm_is_the_references(name, monkeypatch):
    """every level's A (= the reference's R A P), P and R, pattern for pattern and value for value (1e-13)"""
    from saena_b200.sa_setup import build_hierarchy, poisson3d_coo
    monkeypatch.setenv("SAENA_SETUP_SPGEMM", "native")
    g = Golden(name)
    n = round(g.hier.levels[0].A.M ** (1 / 3))
    h = build_hierarchy(*poisson3d_coo(n), device="cuda")
    assert len(h.levels) == len(g.hier.levels)
    for a, b in zip(h.levels, g.hier.levels):
        _same_operator(a.A, b.A)
        if b.P is not None:
            _same_operator(a.P, b.P)
            _same_operator(a.R, b.R)


def test_hierarchy_built_with_the_device_spgemm_is_the_live_references_at_32_cubed(monkeypatch):
    from oracle import ref
    if not ref.available():
        pytest.skip("oracle/_ref/libsaena_ref.so did not travel")
    monkeypatch.setenv("SAENA_SETUP_SPGEMM", "native")
    from saena_b200.sa_setup import build_hierarchy, poisson3d_coo
    s = ref.RefSolver.poisson(34)
    try:
        href = s.hierarchy()
        h = build_hierarchy(*poisson3d_coo(32), device="cuda")
        assert len(h.levels) == len(href.levels)
        for a, b in zip(h.levels, href.levels):
            _same_operator(a.A, b.A)
            if b.P is not None:
                _same_operator(a.P, b.P)
                _same_operator(a.R, b.R)
    finally:
        s.close()


def test_device_spgemm_and_tensor_op_route_build_the_same_64_cubed_hierarchy(monkeypatch):
    """the two product routes of sa_setup.py (device SpGEMM / expand-sort-compress with tensor ops) on a hierarchy with
    1 000-entry rows: same patterns, values to rounding"""
    import torch
    from saena_b200 import sa_setup
    args = sa_setup.poisson3d_coo(64)
    monkeypatch.setenv("SAENA_SETUP_SPGEMM", "native")
    dn = sa_setup.build_device_hierarchy(*args, device="cuda")
    monkeypatch.setenv("SAENA_SETUP_SPGEMM", "torch")
    dt = sa_setup.build_device_hierarchy(*args, device="cuda")
    assert len(dn.levels) == len(dt.levels)
    for a, b in zip(dn.levels, dt.levels):
        assert a.A.nnz == b.A.nnz and torch.equal(a.A.row, b.A.row) and torch.equal(a.A.col, b.A.col)
        assert float((a.A.val - b.A.val).abs().max()) <= 1e-12 * float(b.A.val.abs().max())
