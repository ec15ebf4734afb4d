"""Block solve (saena_b200_solve_pcg_block and its hooks, csrc/spmv_block.cu, the *_block_kernel bodies of
csrc/spmv_kernels.cuh, the block V-cycle of csrc/solve.cu) on the GPU.  Column j of every block call must give, bit for
bit, what the single call gives for column j, one layer at a time: the SpMV with each epilogue on every row mapping
(and the fallback for the mappings without a block body), the operators of a hierarchy, the V-cycle, the PCG solve --
and no column may change another's bits.  Calls the block path refuses leave the single solve as it was."""
import numpy as np
import pytest

from tests import symdiag_cases as sc


def _cuda() -> bool:
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _cuda(), reason="needs a CUDA device")]

KS = (1, 2, 3, 5, 8)


def _same(a, b):
    return np.array_equal(a, b, equal_nan=True)


def _ragged(M=1000, seed=3):
    """rows of 0..40 entries (every 7th row empty), random columns, diagonally dominant where a row has a diagonal"""
    rng = np.random.default_rng(seed)
    rows, cols, vals = [], [], []
    for i in range(M):
        if i % 7 == 3:
            continue
        c = np.unique(np.concatenate([[i], rng.integers(0, M, rng.integers(0, 40))]))
        v = rng.uniform(-1, 0, len(c))
        v[c == i] = 1.0 + np.abs(v).sum()
        rows.append(np.full(len(c), i)), cols.append(c), vals.append(v)
    row, col, val = (np.concatenate(t) for t in (rows, cols, vals))
    rp = np.zeros(M + 1, np.int64)
    np.cumsum(np.bincount(row, minlength=M), out=rp[1:])
    return rp, col.astype(np.int64), val


CASES = {"7pt_37x23x19": lambda: sc.stencil((37, 23, 19), 0, seed=1),    # M = 16169, not a multiple of 32
         "27pt_13x11x9": lambda: sc.stencil((13, 11, 9), 1, seed=2),
         "band8_1500": lambda: sc.band(1500, 8),
         "7pt_3x1x1": lambda: sc.stencil((3, 1, 1), 0, seed=3),           # M = 3 < k
         "ragged_1000": _ragged}                                           # empty rows, irregular lengths
MAPPINGS = [100, 101, 103, 1, 2, 4, 8, 16, 32, 64, 128, 256, -4, "dense"]


def _context(rp, col, val, mapping):
    from saena_b200.hierarchy import F64, I32, KIND_A, Hierarchy, Level, Operator
    from saena_b200.native import Context
    M = len(rp) - 1
    dense = mapping == "dense"
    op = Operator(kind=KIND_A, level=0, M=M, Mbig=M, Nbig=M, row_offset=0, col_offset=0, n_local_cols=M,
                  nnzPerRow_local=np.diff(rp).astype(I32), col_local=col.astype(I32), val_local=val.astype(F64),
                  use_double=not dense, use_dense=dense)
    diag = np.array([val[rp[i]:rp[i + 1]][col[rp[i]:rp[i + 1]] == i].sum() for i in range(M)])
    inv = np.where(diag != 0, 1.0 / np.where(diag != 0, diag, 1.0), 1.0)
    ctx = Context()
    ctx.upload_hierarchy(Hierarchy([Level(0, op, inv_diag=inv, eig_max=1.9)], coarse_n=0))
    if not dense:
        ctx.set_mapping(0, 0, mapping)
    return ctx


def _columns(rng, k, M):
    return rng.uniform(-1, 1, (k, M))


@pytest.mark.parametrize("mapping", MAPPINGS, ids=str)
@pytest.mark.parametrize("name", list(CASES))
def test_kernels_equal_single_calls(name, mapping):
    rp, col, val = CASES[name]()
    M = len(rp) - 1
    ctx = _context(rp, col, val, mapping)
    try:
        rng = np.random.default_rng(7)
        for k in KS:
            x, rhs = _columns(rng, k, M), _columns(rng, k, M)
            got = {"matvec": ctx.matvec_block(0, 0, x), "residual": ctx.residual_block(0, x, rhs),
                   "cheb_zero": ctx.smooth_block(0, "chebyshev", 3, np.zeros_like(x), rhs),
                   "cheb": ctx.smooth_block(0, "chebyshev", 3, x, rhs),
                   "jacobi": ctx.smooth_block(0, "jacobi", 2, x, rhs)}
            for j in range(k):
                want = {"matvec": ctx.matvec(0, 0, x[j]), "residual": ctx.residual(0, x[j], rhs[j]),
                        "cheb_zero": ctx.smooth(0, "chebyshev", 3, np.zeros(M), rhs[j]),
                        "cheb": ctx.smooth(0, "chebyshev", 3, x[j], rhs[j]),
                        "jacobi": ctx.smooth(0, "jacobi", 2, x[j], rhs[j])}
                for key in want:
                    assert _same(got[key][j], want[key]), (name, mapping, k, j, key)
    finally:
        ctx.close()


# ---- hierarchies ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def poisson48():
    import torch
    from saena_b200 import sa_setup
    dh = sa_setup.build_device_hierarchy(*sa_setup.poisson3d_coo(48), device="cuda")
    h = dh.to_rank(0, 1)
    del dh
    torch.cuda.empty_cache()
    assert len(h.levels) >= 3
    return h


@pytest.fixture(scope="module")
def unstructured():
    import torch
    from saena_b200 import sa_setup
    dh = sa_setup.build_device_hierarchy(*sa_setup.unstructured2d_coo(240), device="cuda")
    h = dh.to_rank(0, 1)
    del dh
    torch.cuda.empty_cache()
    assert len(h.levels) >= 3
    return h


def _ctx(h):
    from saena_b200.native import Context
    c = Context()
    c.upload_hierarchy(h)
    return c


def test_every_operator_of_a_hierarchy(poisson48):
    ctx = _ctx(poisson48)
    try:
        rng = np.random.default_rng(1)
        for l, lv in enumerate(poisson48.levels):
            for kind, op in ((0, lv.A), (1, lv.P), (2, lv.R)):
                if op is None:
                    continue
                for k in (2, 3, 8):
                    x = _columns(rng, k, op.n_local_cols)
                    w = ctx.matvec_block(l, kind, x)
                    for j in range(k):
                        assert _same(w[j], ctx.matvec(l, kind, x[j])), (l, kind, k, j)
    finally:
        ctx.close()


def test_dense_flag_hierarchy():
    from tests.util import Golden
    g = Golden("poisson12_dense")
    assert any(lv.A.use_dense for lv in g.hier.levels)
    ctx = _ctx(g.hier)
    try:
        rng = np.random.default_rng(2)
        for l, lv in enumerate(g.hier.levels):
            x = _columns(rng, 3, lv.A.M)
            w = ctx.matvec_block(l, 0, x)
            u = ctx.vcycle_block(l, x, w)
            for j in range(3):
                assert _same(w[j], ctx.matvec(l, 0, x[j])), l
                assert _same(u[j], ctx.vcycle(l, x[j], w[j])), l
        rhs = _columns(rng, 3, g.hier.levels[0].A.M)
        u, iters, hists = ctx.solve_pcg_block(rhs)
        for j in range(3):
            u1, it1, h1 = ctx.solve_pcg(rhs[j])
            assert iters[j] == it1 and _same(hists[j], h1) and _same(u[j], u1)
    finally:
        ctx.close()


@pytest.mark.parametrize("which", ["poisson48", "unstructured"])
def test_vcycle_equals_single_calls(which, request):
    h = request.getfixturevalue(which)
    ctx = _ctx(h)
    try:
        M = h.levels[0].A.M
        rng = np.random.default_rng(4)
        for route in (False, True):
            ctx.set_level_route(1, route)
            for k in (1, 3, 8):
                u0, rhs = _columns(rng, k, M), _columns(rng, k, M)
                got = ctx.vcycle_block(0, u0, rhs)
                zero = ctx.vcycle_block(0, np.zeros_like(u0), rhs, pre=0, post=2, smoother="jacobi")
                for j in range(k):
                    assert _same(got[j], ctx.vcycle(0, u0[j], rhs[j])), (route, k, j)
                    assert _same(zero[j], ctx.vcycle(0, np.zeros(M), rhs[j], pre=0, post=2, smoother="jacobi"))
    finally:
        ctx.close()


# ---- PCG -------------------------------------------------------------------------------------------------------------
def _eight_columns(h):
    from saena_b200 import sa_setup
    M = h.levels[0].A.M
    n = round(M ** (1 / 3))
    rng = np.random.default_rng(2024)
    b = [sa_setup.poisson3d_rhs(n) if n ** 3 == M else rng.standard_normal(M)]
    b += [rng.standard_normal(M) for _ in range(4)]
    b += [3.5 * b[2], b[3].copy(), np.zeros(M)]
    return np.stack(b)


def _check_columns(ctx, rhs, u, iters, hists, **opts):
    for j in range(len(rhs)):
        u1, it1, h1 = ctx.solve_pcg(rhs[j], **opts)
        assert iters[j] == it1, (j, iters[j], it1)
        assert _same(hists[j], h1), j
        assert _same(u[j], u1), j


@pytest.mark.parametrize("graphs", [True, False])
def test_pcg_columns_equal_single_solves(poisson48, graphs):
    ctx = _ctx(poisson48)
    try:
        ctx.set_graphs(graphs)
        rhs = _eight_columns(poisson48)
        u, iters, hists = ctx.solve_pcg_block(rhs)
        _check_columns(ctx, rhs, u, iters, hists)
        assert iters[7] == 1
        # the same columns without the zero one, and with a NaN column in its place: the others keep their bits
        u7, it7, h7 = ctx.solve_pcg_block(rhs[:7])
        bad = rhs.copy()
        bad[7, 5] = np.nan
        un, itn, hn = ctx.solve_pcg_block(bad)
        for j in range(7):
            assert it7[j] == iters[j] == itn[j]
            assert _same(h7[j], hists[j]) and _same(hn[j], hists[j])
            assert _same(u7[j], u[j]) and _same(un[j], u[j])
        assert np.isnan(hn[7][-1])
        # some columns stop at max_iter, the others before
        cap = max(iters) - 1
        u, iters2, hists = ctx.solve_pcg_block(rhs, max_iter=cap)
        assert cap in iters2 and min(iters2) < cap
        _check_columns(ctx, rhs, u, iters2, hists, max_iter=cap)
        # on the route, and replayed again
        ctx.set_level_route(1, True)
        for _ in range(2):
            u, iters, hists = ctx.solve_pcg_block(rhs[:5])
            _check_columns(ctx, rhs[:5], u, iters, hists)
    finally:
        ctx.close()


def test_pcg_after_update_values_and_through_torch(poisson48):
    import torch
    ctx = _ctx(poisson48)
    try:
        A = poisson48.levels[0].A
        rows = np.repeat(np.arange(A.M), A.nnzPerRow_local)
        val = np.where(A.col_local - A.col_offset == rows, A.val_local * 1.2, A.val_local)
        rhs = _eight_columns(poisson48)[:6]
        ctx.solve_pcg_block(rhs)                # block graphs captured before the update
        ctx.update_values(val)
        u, iters, hists = ctx.solve_pcg_block(rhs)
        _check_columns(ctx, rhs, u, iters, hists)
        t = torch.from_numpy(rhs).cuda()
        ud, itd, hd = ctx.solve_pcg_block(t)
        assert ud.is_cuda and itd == iters
        assert all(_same(a, b) for a, b in zip(hd, hists))
        assert _same(ud.cpu().numpy(), u)
    finally:
        ctx.close()


def test_pcg_scaled_hierarchy():
    from tests.util import Golden
    g = Golden("poisson12_cheb")
    h = g.hier
    rng = np.random.default_rng(8)
    h.scale = True
    for lv in h.levels:
        lv.inv_sq_diag = rng.uniform(0.8, 1.25, lv.A.M)
    ctx = _ctx(h)
    try:
        rhs = np.stack([g.rhs, rng.standard_normal(len(g.rhs)), np.zeros(len(g.rhs))])
        u, iters, hists = ctx.solve_pcg_block(rhs)
        _check_columns(ctx, rhs, u, iters, hists)
    finally:
        ctx.close()


def test_refusals_leave_the_single_solve_alone(poisson48):
    from saena_b200 import sa_setup
    from saena_b200.native import Context, NativeError
    ctx = _ctx(poisson48)
    try:
        rhs = _eight_columns(poisson48)
        want = ctx.solve_pcg(rhs[0])
        M = rhs.shape[1]
        for bad in (np.zeros((0, M)), np.zeros((9, M))):
            with pytest.raises(NativeError):
                ctx.solve_pcg_block(bad)
            with pytest.raises(NativeError):
                ctx.matvec_block(0, 0, bad)
            got = ctx.solve_pcg(rhs[0])
            assert got[1] == want[1] and _same(got[2], want[2]) and _same(got[0], want[0])
    finally:
        ctx.close()
    fresh = Context()
    try:
        with pytest.raises(NativeError):
            fresh._ck(fresh._L.saena_b200_matvec_block(fresh._h, 0, 0, 2, None, None))
    finally:
        fresh.close()
    dh = sa_setup.build_device_hierarchy(*sa_setup.poisson3d_coo(16), device="cuda")
    share = Context(rank=0, nranks=2, detached=True)
    try:
        share.upload_hierarchy(dh.to_rank(0, 2))
        with pytest.raises(NativeError):
            share.solve_pcg_block(np.zeros((2, share.level_rows[0])))
        with pytest.raises(NativeError):
            share.vcycle_block(0, np.zeros((2, share.level_rows[0])), np.ones((2, share.level_rows[0])))
    finally:
        share.close()
    ctx = _ctx(poisson48)
    try:
        got = ctx.solve_pcg(rhs[0])
        assert got[1] == want[1] and _same(got[2], want[2]) and _same(got[0], want[0])
    finally:
        ctx.close()
