"""Flexible GMRES (saena_b200_solve_gmres, the Arnoldi kernels of csrc/krylov.cu) on the GPU.

The solve is restated in numpy with the library's own hooks as its building blocks -- ctx.vcycle (ctx.vcycle_f32 at
precision 32) for M^-1 and ctx.matvec for A -- and must reproduce the iterations, the history and u.  The Arnoldi
kernels are covered through the test hook saena_b200_gmres_orthogonalize: every basis size 1..64 against long-double
references within the rounding bound of each entry, and bitwise repeatable.  Then: GMRES's residual is never above
PCG's on SPD hierarchies, nonsymmetric convection-diffusion problems are solved to the tolerance, the edge cases, and
the state the solve shares with the rest of the context."""
import numpy as np
import pytest


def _cuda() -> bool:
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _cuda(), reason="needs a CUDA device")]

JAC = dict(smoother="jacobi", pre=2, post=2)


def _same(a, b):
    return np.array_equal(a, b, equal_nan=True)


# ---- numpy restatement -------------------------------------------------------------------------------------------------
def fgmres_ref(ctx, rhs, restart, max_iter, tol, smoother="chebyshev", pre=3, post=3, bits=64):
    """the header's algorithm step for step: M^-1 through ctx.vcycle / ctx.vcycle_f32 from a zero iterate, A through
    ctx.matvec, CGS2, Givens rotations, u -= Z y, true residual at the end of every cycle"""
    n = len(rhs)
    if bits == 32:
        def prec(v):
            return ctx.vcycle_f32(0, np.zeros(n, np.float32), v.astype(np.float32), pre, post, smoother).astype(np.float64)
    else:
        def prec(v):
            return ctx.vcycle(0, np.zeros(n), v, pre, post, smoother)

    def A(x):
        return ctx.matvec(0, 0, x)

    u = np.zeros(n)
    r = -rhs
    beta = float(np.sqrt(r @ r))
    hist, it = [beta], 0
    if not beta > 0:
        return u, 0, np.array(hist)
    thr = tol * beta
    v = r / beta
    m = restart
    while True:
        V, Z = [v], []
        H = np.zeros((m + 1, m))
        cs, sn, g = np.ones(m), np.zeros(m), np.zeros(m + 1)
        g[0] = beta
        k, nan = 0, False
        for j in range(m):
            if it >= max_iter:
                break
            Z.append(prec(V[j]))
            w = A(Z[j])
            Vm = np.array(V)
            wn = np.sqrt(w @ w)
            h1 = Vm @ w
            w = w - Vm.T @ h1
            h2 = Vm @ w
            w = w - Vm.T @ h2
            hn = np.sqrt(w @ w)
            H[:j + 1, j] = h1 + h2
            it += 1
            k = j + 1
            for i in range(j):
                a, b = H[i, j], H[i + 1, j]
                H[i, j], H[i + 1, j] = cs[i] * a + sn[i] * b, -sn[i] * a + cs[i] * b
            a = H[j, j]
            rr = np.hypot(a, hn)
            cs[j], sn[j] = (a / rr, hn / rr) if rr > 0 else (1.0, 0.0)
            H[j, j] = rr
            g[j + 1] = -sn[j] * g[j]
            g[j] = cs[j] * g[j]
            est = abs(g[j + 1])
            hist.append(est)
            if est != est:
                nan = True
                break
            if not est >= thr or not hn > 0 or hn <= 1e-300 * wn or j + 1 == m or it == max_iter:
                break
            V.append(w / hn)
        if nan:
            break
        y = np.zeros(k)
        for i in range(k - 1, -1, -1):
            s = g[i] - H[i, i + 1:k] @ y[i + 1:k]
            y[i] = s / H[i, i] if H[i, i] != 0 else 0.0
        u = u - np.array(Z[:k]).T @ y
        r = A(u) - rhs
        rn = float(np.sqrt(r @ r))
        if not rn >= thr or it >= max_iter:
            break
        beta = rn
        v = r / beta
    return u, it, np.array(hist)


def _rel(a, b):
    nb = np.linalg.norm(b)
    return np.linalg.norm(a - b) / nb if nb > 0 else np.linalg.norm(a)


def _check_parity(got, want, floor=1e-14, tol_u=1e-10):
    """same iterations; every history entry to 1e-10 relative, above a floor of `floor` ||r0||: an estimate far below
    ||r0|| carries the absolute rounding of the orthogonalisation, some eps ||r0||, whatever the summation order (the
    FP32 preconditioner's floor is wider: an input that differs in its last bits can round to another float)"""
    (u, it, h), (ur, itr, hr) = got, want
    assert it == itr, (it, itr)
    assert len(h) == it + 1 and len(hr) == len(h)
    assert np.all(np.abs(h - hr) <= 1e-10 * np.abs(hr) + floor * hr[0]), np.max(np.abs(h - hr) / hr[0])
    assert _rel(u, ur) <= tol_u, _rel(u, ur)


# ---- hierarchies ---------------------------------------------------------------------------------------------------------
def _ctx(h):
    from saena_b200.native import Context
    c = Context()
    c.upload_hierarchy(h)
    return c


def _csr(op):
    import scipy.sparse as sp
    rp = np.zeros(op.M + 1, np.int64)
    np.cumsum(op.nnzPerRow_local, out=rp[1:])
    return sp.csr_matrix((op.val_local, op.col_local - op.col_offset, rp), shape=(op.M, op.n_local_cols))


_CD = {}


def convdiff(n):
    """hierarchy of the nonsymmetric convection-diffusion operator on n^3 nodes, its matrix and a rhs"""
    if n not in _CD:
        import torch
        from saena_b200 import sa_setup
        N, r, c, v = sa_setup.convdiff3d_coo(n)
        dh = sa_setup.build_device_hierarchy(N, r, c, v, device="cuda")
        h = dh.to_rank(0, 1)
        del dh
        torch.cuda.empty_cache()
        A = _csr(h.levels[0].A)
        assert abs(A - A.T).max() > 0 and len(h.levels) >= 2
        b = np.random.default_rng(n).uniform(-1, 1, N)
        _CD[n] = (h, A, b)
    return _CD[n]


def _golden(name):
    from tests.util import Golden
    g = Golden(name)
    return g.hier, _csr(g.hier.levels[0].A), g.rhs


PROBLEMS = {"poisson9": lambda: _golden("poisson9_cheb"), "poisson12": lambda: _golden("poisson12_cheb"),
            "convdiff16": lambda: convdiff(16), "convdiff32": lambda: convdiff(32), "convdiff48": lambda: convdiff(48)}


def _opts(name):
    # a nonsymmetric level's Chebyshev bound is a heuristic (sa_setup's Lanczos assumes symmetry): Jacobi there
    return JAC if name.startswith("convdiff") else {}


# ---- restatement parity ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(PROBLEMS))
def test_restatement_parity(name):
    h, A, b = PROBLEMS[name]()
    opts = _opts(name)
    ctx = _ctx(h)
    try:
        tol = 1e-9
        u, need, hist = ctx.solve_gmres(b, restart=64, max_iter=300, tol=tol, **opts)
        assert need >= 2
        for restart in (1, 2, 5, need, 64):
            got = ctx.solve_gmres(b, restart=restart, max_iter=300, tol=tol, **opts)
            _check_parity(got, fgmres_ref(ctx, b, restart, 300, tol, **opts))
            assert np.linalg.norm(A @ got[0] - b) <= 10 * tol * np.linalg.norm(b) or got[1] == 300
        # max_iter that is not a multiple of the restart: the last cycle is cut short
        got = ctx.solve_gmres(b, restart=3, max_iter=7, tol=1e-30, **opts)
        assert got[1] == 7
        _check_parity(got, fgmres_ref(ctx, b, 3, 7, 1e-30, **opts))
    finally:
        ctx.close()


@pytest.mark.parametrize("name", ["poisson9", "poisson12", "convdiff32"])
def test_restatement_parity_fp32_preconditioner(name):
    h, A, b = PROBLEMS[name]()
    opts = _opts(name)
    ctx = _ctx(h)
    try:
        ctx.set_precond_precision(32)
        for restart in (5, 30):
            got = ctx.solve_gmres(b, restart=restart, max_iter=200, tol=1e-10, **opts)
            assert got[1] < 200
            assert np.linalg.norm(A @ got[0] - b) <= 1e-9 * np.linalg.norm(b)
            # the Jacobi V-cycle diverges as a stationary iteration on the convection-diffusion hierarchy (it amplifies
            # by ~200 per cycle): there a float that rounds the other way grows out of the rounding floor, and only the
            # solve's own residual is checked
            if name.startswith("poisson"):
                _check_parity(got, fgmres_ref(ctx, b, restart, 200, 1e-10, bits=32, **opts), floor=1e-10, tol_u=1e-8)
    finally:
        ctx.close()


# ---- optimality against PCG -----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def poisson32():
    import torch
    from saena_b200 import sa_setup
    dh = sa_setup.build_device_hierarchy(*sa_setup.poisson3d_coo(32), device="cuda")
    h = dh.to_rank(0, 1)
    del dh
    torch.cuda.empty_cache()
    return h


@pytest.mark.parametrize("name", ["poisson9", "poisson12", "poisson32"])
def test_residual_never_above_pcg(name, request):
    from saena_b200 import sa_setup
    if name == "poisson32":
        h = request.getfixturevalue("poisson32")
        b = sa_setup.poisson3d_rhs(32)
    else:
        h, _, b = PROBLEMS[name]()
    ctx = _ctx(h)
    try:
        for tol, smoother in ((1e-8, "chebyshev"), (1e-10, "chebyshev"), (1e-10, "jacobi")):
            _, itp, hp = ctx.solve_pcg(b, max_iter=100, tol=tol, smoother=smoother)
            _, itg, hg = ctx.solve_gmres(b, restart=max(itp, 1), max_iter=100, tol=tol, smoother=smoother)
            assert itg <= itp, (itg, itp)
            assert abs(hg[0] - hp[0]) <= 1e-14 * hp[0]
            k = min(len(hg), len(hp))
            assert np.all(hg[:k] <= hp[:k] * (1 + 1e-8)), (hg[:k], hp[:k])
    finally:
        ctx.close()


# ---- accuracy on the nonsymmetric problems ---------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [16, 32, 48])
def test_convdiff_accuracy(n):
    import scipy.sparse.linalg as spla
    h, A, b = convdiff(n)
    ctx = _ctx(h)
    try:
        tol = 1e-10
        ref = spla.spsolve(A.tocsc(), b) if n <= 32 else None   # a direct 3-D solve at 48^3 takes minutes
        for restart in (10, 30):
            u, it, hist = ctx.solve_gmres(b, restart=restart, max_iter=300, tol=tol, **JAC)
            assert it < 300
            assert np.linalg.norm(b - A @ u) <= 10 * tol * np.linalg.norm(b)
            assert ref is None or _rel(u, ref) <= 1e4 * tol, _rel(u, ref)
            assert np.all(np.isfinite(hist)) and hist[-1] < tol * hist[0]
    finally:
        ctx.close()


# ---- kernels ---------------------------------------------------------------------------------------------------------------
def test_orthogonalization_kernels_against_long_double():
    from saena_b200.native import Context
    ctx = Context()
    try:
        rng = np.random.default_rng(11)
        L = np.longdouble
        for n in (1, 37, 4099, 70001):
            eps = np.finfo(np.float64).eps
            for nv in list(range(0, 65)) if n == 4099 else (0, 1, 7, 8, 9, 33, 64):
                V = rng.uniform(-1, 1, (nv, n))
                w = rng.uniform(-1, 1, n) + (V.sum(axis=0) * 0.3 if nv else 0)
                w2, h1, h2, col = ctx.gmres_orthogonalize(V, w)
                again = ctx.gmres_orthogonalize(V, w)
                assert all(_same(a, b) for a, b in zip((w2, h1, h2, col), again)), (n, nv)
                g = 2 * (n + 2 * nv + 8) * eps   # the longest chain of roundings of one entry, with a factor 2 to spare
                Vl, wl = V.astype(L), w.astype(L)
                # first pass: h1_i = <v_i, w>, |w|^2
                ref1 = Vl @ wl if nv else np.zeros(0, L)
                assert np.all(np.abs(h1[:nv] - ref1) <= g * (np.abs(V) @ np.abs(w))), (n, nv)
                assert abs(h1[nv] - wl @ wl) <= g * (w @ w)
                # second pass from the device's h1: w' = w - V h1, h2_i = <v_i, w'>
                wp = wl - (Vl.T @ h1[:nv].astype(L) if nv else 0)
                err_wp = g * (np.abs(w) + (np.abs(V).T @ np.abs(h1[:nv]) if nv else 0))
                ref2 = Vl @ wp if nv else np.zeros(0, L)
                bound2 = g * (np.abs(V) @ np.abs(wp.astype(float))) + (np.abs(V) @ err_wp if nv else 0)
                assert np.all(np.abs(h2[:nv] - ref2) <= bound2), (n, nv)
                # final correction from the device's h2: w'' = w' - V h2, ||w''||
                wpp = wp - (Vl.T @ h2[:nv].astype(L) if nv else 0)
                err = err_wp + g * (np.abs(wp.astype(float)) + (np.abs(V).T @ np.abs(h2[:nv]) if nv else 0))
                assert np.all(np.abs(w2 - wpp) <= err), (n, nv)
                assert np.allclose(col[:nv], h1[:nv] + h2[:nv], rtol=0, atol=0)
                assert abs(col[nv] - np.sqrt(float(wpp @ wpp))) <= np.linalg.norm(err) + g * col[nv]
                assert abs(col[nv + 1] - np.sqrt(float(wl @ wl))) <= g * col[nv + 1]
    finally:
        ctx.close()


# ---- edge cases ------------------------------------------------------------------------------------------------------------
def _operator(kind, level, M):
    from saena_b200.hierarchy import F64, I32, Operator
    import scipy.sparse as sp
    M = sp.csr_matrix(M)
    M.sort_indices()
    return Operator(kind=kind, level=level, M=M.shape[0], Mbig=M.shape[0], Nbig=M.shape[1], row_offset=0, col_offset=0,
                    n_local_cols=M.shape[1], nnzPerRow_local=np.diff(M.indptr).astype(I32),
                    col_local=M.indices.astype(I32), val_local=M.data.astype(F64))


def _two_level(A0, P, inv_diag):
    """level 0's A, P, R = P^T and the exact coarsest level R A P"""
    import scipy.sparse as sp
    from saena_b200.hierarchy import Hierarchy, Level
    A0, P = sp.csr_matrix(A0), sp.csr_matrix(P)
    R = P.T.tocsr()
    Ac = (R @ A0 @ P).tocoo()
    lv0 = Level(0, _operator(0, 0, A0), inv_diag=np.asarray(inv_diag, float), eig_max=2.0, P=_operator(1, 0, P),
                R=_operator(2, 0, R), M_coarse_old=P.shape[1], M_coarse=P.shape[1])
    lv1 = Level(1, _operator(0, 1, Ac.tocsr()), inv_diag=1.0 / Ac.tocsr().diagonal(), eig_max=2.0)
    return Hierarchy([lv0, lv1], coarse_n=P.shape[1], coarse_row=Ac.row.astype(np.int32),
                     coarse_col=Ac.col.astype(np.int32), coarse_val=Ac.data)


def test_breakdown_at_step_three():
    # A = diag(1, 2, 4) under a V-cycle with an unscaled Jacobi (inv_diag = 1) and a rank-one coarse space: the
    # preconditioned operator is a 3 x 3 matrix with three distinct eigenvalues, so the Krylov space is complete at
    # step 3 and h_{3,2} vanishes (to rounding)
    A0 = np.diag([1.0, 2.0, 4.0])
    h = _two_level(A0, np.ones((3, 1)), np.ones(3))
    ctx = _ctx(h)
    try:
        b = np.array([1.0, -2.0, 0.5])
        for restart in (3, 10, 64):
            u, it, hist = ctx.solve_gmres(b, restart=restart, max_iter=20, tol=1e-12, **JAC)
            assert it == 3, (restart, it, hist)
            assert np.all(np.isfinite(hist)) and np.all(np.isfinite(u))
            assert np.linalg.norm(u - b / np.diag(A0)) <= 1e-10 * np.linalg.norm(u)
            _check_parity((u, it, hist), fgmres_ref(ctx, b, restart, 20, 1e-12, **JAC))
    finally:
        ctx.close()


def test_zero_and_nan_rhs():
    h, A, b = _golden("poisson9_cheb")
    ctx = _ctx(h)
    try:
        want = ctx.solve_gmres(b, restart=10)
        u, it, hist = ctx.solve_gmres(np.zeros_like(b), restart=10)
        assert it == 0 and len(hist) == 1 and hist[0] == 0.0
        assert _same(u, np.zeros_like(b))
        bad = b.copy()
        bad[3] = np.nan
        u, it, hist = ctx.solve_gmres(bad, restart=10)
        assert it == 0 and len(hist) == 1 and np.isnan(hist[0])
        _, itp, hp = ctx.solve_pcg(bad)
        assert np.isnan(hp[-1])   # PCG stops at its first NaN too
        # nothing carries over into the next solve
        got = ctx.solve_gmres(b, restart=10)
        assert got[1] == want[1] and _same(got[2], want[2]) and _same(got[0], want[0])
    finally:
        ctx.close()


def test_one_level_takes_the_direct_path():
    import scipy.sparse as sp
    from saena_b200.hierarchy import Hierarchy, Level
    from saena_b200 import sa_setup
    N, r, c, v = sa_setup.convdiff3d_coo(6)
    A = sp.csr_matrix((v, (r, c)), shape=(N, N))
    coo = A.tocoo()
    h = Hierarchy([Level(0, _operator(0, 0, A), inv_diag=1.0 / A.diagonal(), eig_max=2.0)], coarse_n=N,
                  coarse_row=coo.row.astype(np.int32), coarse_col=coo.col.astype(np.int32), coarse_val=coo.data)
    ctx = _ctx(h)
    try:
        b = np.random.default_rng(5).uniform(-1, 1, N)
        u, it, hist = ctx.solve_gmres(b, restart=5, tol=1e-12)
        assert it == 1 and len(hist) == 2
        assert np.linalg.norm(A @ u - b) <= 1e-12 * np.linalg.norm(b)
        assert hist[1] <= 1e-12 * hist[0]
    finally:
        ctx.close()


# ---- state -----------------------------------------------------------------------------------------------------------------
def test_graphs_repeats_and_other_solvers():
    h, A, b = convdiff(32)
    ctx = _ctx(h)
    try:
        pcg = ctx.solve_pcg(b, **JAC)
        blk = ctx.solve_pcg_block(np.stack([b, -b]), **JAC)
        first = ctx.solve_gmres(b, restart=5, **JAC)
        for graphs in (True, False, True):
            ctx.set_graphs(graphs)
            for _ in range(2):
                got = ctx.solve_gmres(b, restart=5, **JAC)
                assert got[1] == first[1] and _same(got[2], first[2]) and _same(got[0], first[0])
        # growing the restart, then back
        ctx.solve_gmres(b, restart=40, **JAC)
        got = ctx.solve_gmres(b, restart=5, **JAC)
        assert got[1] == first[1] and _same(got[2], first[2]) and _same(got[0], first[0])
        # PCG and block PCG keep their bits
        p2 = ctx.solve_pcg(b, **JAC)
        assert p2[1] == pcg[1] and _same(p2[2], pcg[2]) and _same(p2[0], pcg[0])
        b2 = ctx.solve_pcg_block(np.stack([b, -b]), **JAC)
        assert b2[1] == blk[1] and _same(b2[0], blk[0]) and all(_same(x, y) for x, y in zip(b2[2], blk[2]))
        # the device-pointer entry gives the host entry's bits
        import torch
        t = torch.from_numpy(b).cuda()
        ud = torch.zeros_like(t)
        torch.cuda.synchronize()
        itd, hd = ctx.solve_gmres_dev(t.data_ptr(), ud.data_ptr(), restart=5, **JAC)
        assert itd == first[1] and _same(hd, first[2]) and _same(ud.cpu().numpy(), first[0])
    finally:
        ctx.close()


def test_after_state_changes(poisson32):
    from saena_b200 import sa_setup
    h = poisson32
    b = sa_setup.poisson3d_rhs(32)
    A = _csr(h.levels[0].A)
    ctx = _ctx(h)

    def check(Am, bits=64):
        got = ctx.solve_gmres(b, restart=10, tol=1e-10)
        assert np.linalg.norm(Am @ got[0] - b) <= 1e-9 * np.linalg.norm(b)
        if bits == 32:
            _check_parity(got, fgmres_ref(ctx, b, 10, 100, 1e-10, bits=32), floor=1e-10, tol_u=1e-8)
        else:
            _check_parity(got, fgmres_ref(ctx, b, 10, 100, 1e-10))

    try:
        ctx.set_precond_precision(32)
        check(A, 32)
        rows = np.repeat(np.arange(A.shape[0]), h.levels[0].A.nnzPerRow_local)
        val = np.where(h.levels[0].A.col_local == rows, h.levels[0].A.val_local * 1.3, h.levels[0].A.val_local)
        ctx.update_values(val)
        A2 = A.copy()
        A2.setdiag(A.diagonal() * 1.3)
        check(A2, 32)
        ctx.set_mapping(0, 0, 100)
        check(A2, 32)
        ctx.set_level_route(1, True)
        check(A2, 32)
        ctx.set_precond_precision(64)
        check(A2)
    finally:
        ctx.close()


def test_refusals_leave_the_context_usable():
    from saena_b200 import sa_setup
    from saena_b200.native import Context, NativeError
    h, A, b = _golden("poisson9_cheb")
    ctx = _ctx(h)
    try:
        want = ctx.solve_gmres(b, restart=10)
        for kw in (dict(restart=0), dict(restart=65), dict(max_iter=0), dict(restart=-3)):
            with pytest.raises(NativeError):
                ctx.solve_gmres(b, **kw)
            got = ctx.solve_gmres(b, restart=10)
            assert got[1] == want[1] and _same(got[2], want[2]) and _same(got[0], want[0])
            pcg = ctx.solve_pcg(b)
            assert pcg[1] > 0
    finally:
        ctx.close()
    fresh = Context()
    try:
        with pytest.raises(NativeError):
            fresh._ck(fresh._L.saena_b200_solve_gmres(fresh._h, None, None, 10, 10, 1e-8, 1, 3, 3, None, None, 0, None))
    finally:
        fresh.close()
    dh = sa_setup.build_device_hierarchy(*sa_setup.poisson3d_coo(16), device="cuda")
    share = Context(rank=0, nranks=2, detached=True)
    try:
        share.upload_hierarchy(dh.to_rank(0, 2))
        with pytest.raises(NativeError):
            share.solve_gmres(np.ones(share.level_rows[0]))
    finally:
        share.close()
