"""FP32 preconditioner (saena_b200_set_precond_precision 32, csrc/spmv_f32.cu, the float instantiations of the
spmv_kernels.cuh bodies and of the V-cycle in csrc/solve.cu) on the GPU.  The FP32 kernels are checked against the FP64
ones fed float-rounded values and inputs, row by row, within the rounding of a float sum; the FP32 V-cycle against the
FP64 one; PCG with the FP32 preconditioner against FP64 PCG in iterations and true residual.  Switching to 32 and back
changes no FP64 bit, the FP32 copies follow every call that changes values or layouts, and the refusals leave the
context at 64."""
import numpy as np
import pytest
import scipy.sparse as sp

from tests.test_zz_block_solve_gpu import CASES


def _cuda() -> bool:
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _cuda(), reason="needs a CUDA device")]

U = 2.0 ** -24
F32 = np.float32
MAPPINGS = [100, 101, 103, 1, 2, 4, 8, 16, 32, 64, 128, 256, "dense"]


def _same(a, b):
    return np.array_equal(a, b, equal_nan=True)


def _r32(a):
    return np.asarray(a, np.float64).astype(F32).astype(np.float64)


def _csr(op):
    rp = np.zeros(op.M + 1, np.int64)
    np.cumsum(op.nnzPerRow_local, out=rp[1:])
    return sp.csr_matrix((op.val_local, op.col_local - op.col_offset, rp), shape=(op.M, op.n_local_cols))


def _gamma(A):
    """per row: 4 len_i 2^-24 -- the rounding of a float sum of len_i products, values rounded to float"""
    return 4.0 * np.diff(A.indptr) * U


def _within(got, want, bound, what):
    err = np.abs(np.asarray(got, np.float64) - want)
    bad = np.flatnonzero(err > bound * (1 + 1e-6) + 1e-37)
    assert bad.size == 0, (what, bad[:5], err[bad[:5]], bound[bad[:5]])


def _context(rp, col, val, mapping):
    """one level-0 operator with float-rounded values and inv_diag, so that the FP64 hooks see what the FP32 ones do"""
    from saena_b200.hierarchy import F64, I32, KIND_A, Hierarchy, Level, Operator
    from saena_b200.native import Context
    M = len(rp) - 1
    dense = mapping == "dense"
    val = _r32(val)
    op = Operator(kind=KIND_A, level=0, M=M, Mbig=M, Nbig=M, row_offset=0, col_offset=0, n_local_cols=M,
                  nnzPerRow_local=np.diff(rp).astype(I32), col_local=col.astype(I32), val_local=val.astype(F64),
                  use_double=not dense, use_dense=dense)
    diag = np.array([val[rp[i]:rp[i + 1]][col[rp[i]:rp[i + 1]] == i].sum() for i in range(M)])
    inv = _r32(np.where(diag != 0, 1.0 / np.where(diag != 0, diag, 1.0), 1.0))
    ctx = Context()
    ctx.upload_hierarchy(Hierarchy([Level(0, op, inv_diag=inv, eig_max=1.9)], coarse_n=0))
    if not dense:
        ctx.set_mapping(0, 0, mapping)
    ctx.set_precond_precision(32)
    A = sp.csr_matrix((val, col, rp), shape=(M, M))
    return ctx, A, inv


@pytest.mark.parametrize("mapping", MAPPINGS, ids=str)
@pytest.mark.parametrize("name", list(CASES))
def test_kernels_within_float_rounding(name, mapping):
    rp, col, val = CASES[name]()
    ctx, A, inv = _context(rp, col, val, mapping)
    try:
        M = A.shape[0]
        rng = np.random.default_rng(11)
        x, rhs = _r32(rng.uniform(-1, 1, M)), _r32(rng.uniform(-1, 1, M))
        g = _gamma(A)
        S = abs(A) @ np.abs(x)                       # sum_j |a_ij x_j|
        ax = ctx.matvec(0, 0, x)
        theta = (1.9 + 0.13 * 1.9) / 2.0
        omega = float(F32(2.0 / 3))
        runs = {
            "matvec": (lambda: ctx.matvec_f32(0, 0, x.astype(F32)), ax, g * S + U * np.abs(ax)),
            "residual": (lambda: ctx.residual_f32(0, x.astype(F32), rhs.astype(F32)), ctx.residual(0, x, rhs),
                         g * S + 2 * U * (np.abs(ax) + np.abs(rhs))),
            "cheb_zero": (lambda: ctx.smooth_f32(0, "chebyshev", 1, np.zeros(M, F32), rhs.astype(F32)),
                          ctx.smooth(0, "chebyshev", 1, np.zeros(M), rhs), 4 * U * np.abs(inv * rhs / theta)),
            "cheb": (lambda: ctx.smooth_f32(0, "chebyshev", 1, x.astype(F32), rhs.astype(F32)),
                     ctx.smooth(0, "chebyshev", 1, x, rhs),
                     np.abs(inv / theta) * (g * S + 4 * U * (np.abs(ax) + np.abs(rhs))) + 4 * U * (
                         np.abs(x) + np.abs(inv * (rhs - ax) / theta))),
            "jacobi": (lambda: ctx.smooth_f32(0, "jacobi", 1, x.astype(F32), rhs.astype(F32)),
                       ctx.smooth(0, "jacobi", 1, x, rhs),
                       np.abs(inv * omega) * (g * S + 4 * U * (np.abs(ax) + np.abs(rhs))) + 4 * U * (
                           np.abs(x) + np.abs(inv * omega * (ax - rhs)))),
        }
        for key, (run, want, bound) in runs.items():
            got = run()
            assert got.dtype == F32
            _within(got, want, bound, (name, mapping, key))
            assert _same(run(), got), (name, mapping, key)    # the same bits twice
        # several Chebyshev sweeps from zero: a relative check
        got = ctx.smooth_f32(0, "chebyshev", 3, np.zeros(M, F32), rhs.astype(F32))
        want = ctx.smooth(0, "chebyshev", 3, np.zeros(M), rhs)
        assert np.linalg.norm(got - want) <= 1e-5 * max(np.linalg.norm(want), 1e-30), (name, mapping)
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


def _ctx(h, bits=64):
    from saena_b200.native import Context
    c = Context()
    c.upload_hierarchy(h)
    if bits == 32:
        c.set_precond_precision(32)
    return c


def _rhs(h, seed=2024):
    from saena_b200 import sa_setup
    M = h.levels[0].A.M
    n = round(M ** (1 / 3))
    return sa_setup.poisson3d_rhs(n) if n ** 3 == M else np.random.default_rng(seed).standard_normal(M)


def test_every_operator_and_the_vcycle_of_a_hierarchy(poisson48):
    h = poisson48
    ctx = _ctx(h, 32)
    try:
        rng = np.random.default_rng(1)
        for route in (False, True):
            ctx.set_level_route(1, route)
            for l, lv in enumerate(h.levels):
                for kind, op in ((0, lv.A), (1, lv.P), (2, lv.R)):
                    if op is None:
                        continue
                    x = _r32(rng.uniform(-1, 1, op.n_local_cols))
                    A = _csr(op)
                    want = ctx.matvec(l, kind, x)
                    if kind == 0 and l == 1 and route:
                        # R (A (P x)): each stage's rounding carried through the absolute values of the next ones
                        fl = h.levels[0]
                        P, A0, R = _csr(fl.P), _csr(fl.A), _csr(fl.R)
                        S = abs(R) @ (abs(A0) @ (abs(P) @ np.abs(x)))
                        lens = np.diff(R.indptr) + np.diff(A0.indptr).max() + np.diff(P.indptr).max() + 3
                        bound = 4 * U * lens * S
                    else:
                        bound = _gamma(A) * (abs(A) @ np.abs(x)) + U * np.abs(want)
                    _within(ctx.matvec_f32(l, kind, x.astype(F32)), want, bound, (route, l, kind))
            M = h.levels[0].A.M
            for smoother in ("chebyshev", "jacobi"):
                rhs = rng.standard_normal(M)
                want = ctx.vcycle(0, np.zeros(M), rhs, smoother=smoother)
                got = ctx.vcycle_f32(0, np.zeros(M, F32), rhs.astype(F32), smoother=smoother)
                assert np.linalg.norm(got - want) <= 1e-5 * np.linalg.norm(want), (route, smoother)
    finally:
        ctx.close()


# ---- PCG -------------------------------------------------------------------------------------------------------------
def _true_residual(ctx, b, u):
    return np.linalg.norm(ctx.residual(0, u, b)) / np.linalg.norm(b)


@pytest.mark.parametrize("smoother", ["chebyshev", "jacobi"])
@pytest.mark.parametrize("which", ["poisson48", "unstructured"])
def test_pcg_iterations_and_true_residual(which, smoother, request):
    h = request.getfixturevalue(which)
    b = _rhs(h)
    tol = 1e-8
    c64, c32 = _ctx(h), _ctx(h, 32)
    try:
        u64, it64, h64 = c64.solve_pcg(b, tol=tol, smoother=smoother)
        u32, it32, h32 = c32.solve_pcg(b, tol=tol, smoother=smoother)
        assert it32 <= it64 + 1, (which, smoother, it64, it32, h64, h32)
        assert _true_residual(c64, b, u32) <= 2 * tol, (which, smoother)
        again = c32.solve_pcg(b, tol=tol, smoother=smoother)
        assert again[1] == it32 and _same(again[2], h32) and _same(again[0], u32)
        c32.set_graphs(False)
        eager = c32.solve_pcg(b, tol=tol, smoother=smoother)
        assert eager[1] == it32 and _same(eager[2], h32) and _same(eager[0], u32)
    finally:
        c64.close()
        c32.close()


def test_pcg_through_the_device_pointer_entry(poisson48):
    import torch
    b = _rhs(poisson48)
    ctx = _ctx(poisson48, 32)
    try:
        u, it, hist = ctx.solve_pcg(b)
        bt = torch.from_numpy(b).cuda()
        ut = torch.zeros_like(bt)
        itd, histd = ctx.solve_pcg_dev(bt.data_ptr(), ut.data_ptr())
        assert itd == it and _same(histd, hist) and _same(ut.cpu().numpy(), u)
    finally:
        ctx.close()


def test_nothing_changes_at_64(poisson48):
    b = _rhs(poisson48)
    fresh = _ctx(poisson48)
    ctx = _ctx(poisson48)
    try:
        others = {name: getattr(ctx, name)(b, max_iter=4) for name in ("solve_vcycle", "solve_cg", "solve_smoother")}
        want = fresh.solve_pcg(b)
        ctx.set_precond_precision(32)
        assert ctx.get_precond_precision() == 32
        for name, w in others.items():   # the switch is ignored by these
            g = getattr(ctx, name)(b, max_iter=4)
            assert g[1] == w[1] and _same(g[2], w[2]) and _same(g[0], w[0]), name
        ctx.solve_pcg(b)
        ctx.set_precond_precision(64)
        assert ctx.get_precond_precision() == 64
        got = ctx.solve_pcg(b)
        assert got[1] == want[1] and _same(got[2], want[2]) and _same(got[0], want[0])
    finally:
        fresh.close()
        ctx.close()


# ---- staleness -------------------------------------------------------------------------------------------------------
def _asymmetric_values(op):
    rows = np.repeat(np.arange(op.M), op.nnzPerRow_local)
    val = np.where(op.col_local - op.col_offset == rows, op.val_local * 1.2, op.val_local)
    off = np.flatnonzero(op.col_local - op.col_offset != rows)[0]
    val[off] *= 1.0 + 2.0 ** -40          # one entry off its mirror: level 0 leaves the symmetric diagonals
    return val


def _scaled_diagonal(op):
    rows = np.repeat(np.arange(op.M), op.nnzPerRow_local)
    return np.where(op.col_local - op.col_offset == rows, op.val_local * 1.2, op.val_local)


def _copy_configuration(src, dst, h):
    """mappings and routes of src onto dst"""
    for l, lv in enumerate(h.levels):
        for kind, op in ((0, lv.A), (1, lv.P), (2, lv.R)):
            if op is not None and dst.get_mapping(l, kind) != src.get_mapping(l, kind):
                dst.set_mapping(l, kind, src.get_mapping(l, kind))
    for l in range(1, len(h.levels)):
        if src.get_level_route(l) != dst.get_level_route(l):
            dst.set_level_route(l, src.get_level_route(l))


CHANGES = {
    "update_values": lambda c, h: c.update_values(_scaled_diagonal(h.levels[0].A)),
    "update_leaves_103": lambda c, h: c.update_values(_asymmetric_values(h.levels[0].A)),
    "set_mapping": lambda c, h: c.set_mapping(1, 0, 101),
    "autotune_mapping": lambda c, h: c.autotune_mapping_native(reps=3),
    "set_level_route": lambda c, h: c.set_level_route(1, True),
    "set_coarsest_solver": lambda c, h: c.set_coarsest_solver("CG"),
}


@pytest.mark.parametrize("change", list(CHANGES))
def test_copies_follow_every_change(poisson48, change):
    h = poisson48
    b = _rhs(h)
    before, after = _ctx(h), _ctx(h)
    try:
        for c in (before, after):
            c.set_mapping(0, 0, 103)
            assert c.get_mapping(0, 0) == 103
        CHANGES[change](before, h)
        after.set_precond_precision(32)
        after.solve_pcg(b)                   # copies and graphs of the old state exist
        CHANGES[change](after, h)
        if change == "autotune_mapping":     # chosen by timing: give `before` what `after` chose
            _copy_configuration(after, before, h)
        if change == "update_leaves_103":
            assert after.get_mapping(0, 0) != 103 and before.get_mapping(0, 0) != 103
        before.set_precond_precision(32)
        want, got = before.solve_pcg(b), after.solve_pcg(b)
        assert got[1] == want[1] and _same(got[2], want[2]) and _same(got[0], want[0]), change
    finally:
        before.close()
        after.close()


# ---- refusals --------------------------------------------------------------------------------------------------------
def test_refusals_leave_the_context_at_64(poisson48):
    from saena_b200 import sa_setup
    from saena_b200.native import Context, NativeError
    from tests.util import Golden
    b = _rhs(poisson48)
    ctx = _ctx(poisson48)
    try:
        want = ctx.solve_pcg(b)

        def unchanged():
            assert ctx.get_precond_precision() == 64
            got = ctx.solve_pcg(b)
            assert got[1] == want[1] and _same(got[2], want[2]) and _same(got[0], want[0])

        for bits in (0, 16, 63):
            with pytest.raises(NativeError):
                ctx.set_precond_precision(bits)
            unchanged()
        with pytest.raises(NativeError):     # the FP32 hooks at 64
            ctx.matvec_f32(0, 0, np.zeros(b.size, F32))
        # streaming row blocks: refused at the switch, and at the next FP32 solve after the switch
        ctx.set_mapping(0, 0, -4)
        with pytest.raises(NativeError):
            ctx.set_precond_precision(32)
        assert ctx.get_precond_precision() == 64
        ctx.set_mapping(0, 0, 0)
        unchanged()
        ctx.set_precond_precision(32)
        ctx.set_mapping(1, 0, -4)
        with pytest.raises(NativeError):
            ctx.solve_pcg(b)
        assert ctx.get_precond_precision() == 64
        ctx.set_mapping(1, 0, 0)
        unchanged()
        # the block solve refuses at 32 and works again at 64
        ctx.set_precond_precision(32)
        with pytest.raises(NativeError):
            ctx.solve_pcg_block(np.stack([b, b]))
        with pytest.raises(NativeError):
            ctx.matvec_block(0, 0, np.zeros((2, b.size)))
        ctx.set_precond_precision(64)
        u, iters, hists = ctx.solve_pcg_block(np.stack([b, b]))
        assert iters == [want[1]] * 2 and _same(u[0], want[0])
        unchanged()
    finally:
        ctx.close()
    fresh = Context()                         # not finalized
    try:
        with pytest.raises(NativeError):
            fresh.set_precond_precision(32)
        assert fresh.get_precond_precision() == 64
    finally:
        fresh.close()
    g = Golden("poisson12_cheb")              # a scaled hierarchy
    hs = g.hier
    rng = np.random.default_rng(8)
    hs.scale = True
    for lv in hs.levels:
        lv.inv_sq_diag = rng.uniform(0.8, 1.25, lv.A.M)
    scaled = _ctx(hs)
    try:
        w = scaled.solve_pcg(g.rhs)
        with pytest.raises(NativeError):
            scaled.set_precond_precision(32)
        got = scaled.solve_pcg(g.rhs)
        assert scaled.get_precond_precision() == 64 and got[1] == w[1] and _same(got[0], w[0])
    finally:
        scaled.close()
    dh = sa_setup.build_device_hierarchy(*sa_setup.poisson3d_coo(16), device="cuda")
    share = Context(rank=0, nranks=2, detached=True)   # several ranks, a detached share
    try:
        share.upload_hierarchy(dh.to_rank(0, 2))
        with pytest.raises(NativeError):
            share.set_precond_precision(32)
        assert share.get_precond_precision() == 64
    finally:
        share.close()
