"""Parity tests proper: the CUDA path, called through the C ABI (saena_b200.native -> include/
saena_b200.h), against (1) the golden vectors the reference wrote, (2) the CPU oracle on the same
seeded inputs, (3) the compiled reference itself where oracle/_ref travelled with the snapshot.
Tolerances are the north_star's: 1e-12 relative per SpMV / smoother sweep / transfer, iteration
count +-1, residual-norm history 1e-9."""
import numpy as np
import pytest

from oracle.oracle import Oracle
from saena_b200.hierarchy import KIND_A, KIND_P, KIND_R, Hierarchy, Level, Operator
from saena_b200.native import Context
from tests.util import (GOLDEN, GOLDEN_EXTRA, TOL_HIST, TOL_OP, Golden, check_ops_against_golden, check_pcg,
                        check_vcycle_against_golden, rel)

pytestmark = pytest.mark.gpu

MAPPINGS = [0, 1, 2, 4, 8, 16, 32, 64, 128, 256, -1, -2, -4, -8, -16, -32, 100]


@pytest.fixture(scope="module", params=GOLDEN)
def golden_ctx(request):
    g = Golden(request.param)
    ctx = Context()
    ctx.upload_hierarchy(g.hier)
    yield g, ctx
    ctx.close()


def test_ops_match_reference_golden(golden_ctx):
    g, ctx = golden_ctx
    check_ops_against_golden(ctx, g)


def test_vcycle_matches_reference_golden(golden_ctx):
    g, ctx = golden_ctx
    check_vcycle_against_golden(ctx, g)


def test_pcg_matches_reference_golden(golden_ctx):
    g, ctx = golden_ctx
    u, iters, hist = ctx.solve_pcg(g.rhs, g.max_iter, g.tol, "chebyshev", g.pre, g.post)
    check_pcg(iters, hist, u, int(g["out.pcg.iters"][0]), g["out.pcg.hist"], g["out.pcg.u"])
    A = g.hier.levels[0].A.to_scipy_local()
    assert np.linalg.norm(A @ u - g.rhs) / np.linalg.norm(g.rhs) < g.tol
    assert ctx.launch_count() > 0


@pytest.mark.parametrize("name", GOLDEN_EXTRA)
def test_other_matrix_shapes_match_reference_golden(name):
    """irregular rows (Helmholtz2D, configs[4]'s shape), a system PCG does not converge on (homg: the
    whole 50-iteration history must still match), the band pattern of configs[3] (operators only)"""
    g = Golden(name)
    ctx = Context()
    try:
        ctx.upload_hierarchy(g.hier)
        check_ops_against_golden(ctx, g)
        check_vcycle_against_golden(ctx, g)
        for mp in (1, 8, 64, -4, 100, 0):   # and through the other row mappings
            for l, lv in enumerate(g.hier.levels):
                ctx.set_mapping(l, KIND_A, mp)
                assert rel(ctx.matvec(l, KIND_A, g[f"in.L{l}.v"]), g[f"out.L{l}.A_matvec"]) <= TOL_OP, (name, mp, l)
        if g.has_pcg:
            u, iters, hist = ctx.solve_pcg(g.rhs, g.max_iter, g.tol, "chebyshev", g.pre, g.post)
            check_pcg(iters, hist, u, int(g["out.pcg.iters"][0]), g["out.pcg.hist"], g["out.pcg.u"])
    finally:
        ctx.close()


@pytest.mark.parametrize("g,lengths,weights", [(160, (6, 8, 10), (16, 48, 20)), (72, (24, 32, 40), (64, 192, 80))])
def test_unstructured_helmholtz_like_shape_matches_oracle(g, lengths, weights):
    """BASELINE.json configs[4]'s synthetic shape at a size the oracle finishes in seconds: irregular
    rows, mesh-like numbering; every operator, V-cycle and the PCG history against the CPU oracle"""
    from saena_b200.sa_setup import build_hierarchy, unstructured2d_coo, unstructured2d_rhs
    n, row, col, val = unstructured2d_coo(g, row_lengths=lengths, weights=weights)
    rhs = unstructured2d_rhs(n)
    h = build_hierarchy(n, row, col, val, device="cpu")
    o = Oracle(h)
    ctx = Context()
    rng = np.random.default_rng(11)
    try:
        ctx.upload_hierarchy(h)
        for l, lv in enumerate(h.levels):
            v, b = rng.uniform(-1, 1, lv.A.M), rng.uniform(-1, 1, lv.A.M)
            assert rel(ctx.matvec(l, KIND_A, v), o.matvec(l, KIND_A, v)) <= TOL_OP
            assert rel(ctx.smooth(l, "chebyshev", 3, v, b), o.smooth(l, "chebyshev", 3, v, b)) <= TOL_OP
            assert rel(ctx.smooth(l, "jacobi", 2, v, b), o.smooth(l, "jacobi", 2, v, b)) <= TOL_OP
            if lv.P is not None:
                vc = rng.uniform(-1, 1, lv.P.n_local_cols)
                assert rel(ctx.matvec(l, KIND_P, vc), o.matvec(l, KIND_P, vc)) <= TOL_OP
                assert rel(ctx.matvec(l, KIND_R, v), o.matvec(l, KIND_R, v)) <= TOL_OP
            assert rel(ctx.vcycle(l, np.zeros(lv.A.M), b), o.vcycle(l, np.zeros(lv.A.M), b)) <= 1e-11
        u, iters, hist = ctx.solve_pcg(rhs, 50, 1e-8, "chebyshev", 3, 3)
        u_o, it_o, h_o = o.solve_pcg(rhs, 50, 1e-8, "chebyshev", 3, 3)
        check_pcg(iters, hist, u, it_o, h_o, u_o)
    finally:
        ctx.close()


@pytest.mark.parametrize("name", ["poisson9_cheb", "poisson12_cheb", "helmholtz2d_p8"])
def test_find_eig_on_device_matches_reference_engine(name):
    """SURVEY 8f #1 (saena_object::find_eig on the device): same start vectors as the reference's own
    Lanczos engine was given (tests/golden/find_eig.npz) -> same bound, same number of steps; the
    seeded generator gives the stored bound up to the start-vector dependence; installing the result
    keeps the solve converging"""
    import os
    from tests.util import GOLDEN_DIR
    d = np.load(os.path.join(GOLDEN_DIR, "find_eig.npz"))
    g = Golden(name)
    ctx = Context()
    try:
        ctx.upload_hierarchy(g.hier)
        for l, lv in enumerate(g.hier.levels):
            eig, iters = ctx.find_eig(l, start=d[f"{name}.L{l}.start"])
            want = float(d[f"{name}.L{l}.eig"][0])
            assert abs(eig - want) <= 5e-9 * want, (name, l, eig, want)
            assert abs(iters - int(d[f"{name}.L{l}.iters"][0])) <= 1, (name, l, iters)
            eig_s, _ = ctx.find_eig(l, seed=42)
            assert abs(eig_s - lv.eig_max) <= 2e-2 * lv.eig_max, (name, l, eig_s, lv.eig_max)
            assert ctx.find_eig(l, seed=42)[0] == eig_s          # reproducible
        u0, it0, h0 = ctx.solve_pcg(g.rhs, g.max_iter, g.tol)
        for l in range(len(g.hier.levels)):
            ctx.find_eig(l, seed=7, store=True)
        u1, it1, h1 = ctx.solve_pcg(g.rhs, g.max_iter, g.tol)
        assert abs(it1 - it0) <= 1 and h1[-1] < h1[0] * g.tol
    finally:
        ctx.close()


def _band_rows(n, b, v, rows):
    """(A v)_i of the band matrix for a few rows, summed in column order like the kernels' CSR order"""
    out = []
    for i in rows:
        j = np.arange(max(i - b, 0), min(i + b, n - 1) + 1)
        out.append(float(np.sum(v[j] / (i + j + 1.0))))
    return np.array(out)


@pytest.mark.parametrize("n,b", [(1, 0), (50, 3), (5000, 40), (4097, 64), (70, 64)])
def test_device_generated_band_operator(n, b):
    """saena_b200_upload_band_operator (the configs[3] measurement input) against the band matrix
    written out row by row, through every mapping; and against the reference's own matvec on the
    same pattern (golden band8_1500)"""
    rng = np.random.default_rng(5)
    v = rng.uniform(-1, 1, n)
    ctx = Context()
    try:
        nnz = ctx.upload_band(n, b)
        assert nnz == sum(min(i + b, n - 1) - max(i - b, 0) + 1 for i in range(n))
        want = _band_rows(n, b, v, range(n))
        for mp in (0, 1, 4, 32, 256, -2, 100):
            ctx.set_mapping(0, KIND_A, mp)
            assert rel(ctx.matvec(0, KIND_A, v), want) <= TOL_OP, (n, b, mp)
        # one fused Chebyshev sweep = u + (1/theta) D^-1 (rhs - A u) with D^-1 = 2i+1, eig_max 2.0
        if n >= 50:
            # the full-size configuration keeps only the sliced copy (CSR entries released)
            ctx.upload_band(n, b, sliced_only=True)
            assert ctx.get_mapping(0, KIND_A) == 100
            assert rel(ctx.matvec(0, KIND_A, v), want) <= TOL_OP
            with pytest.raises(Exception, match="sliced copy"):
                ctx.set_mapping(0, KIND_A, 8)
        rhs = rng.uniform(-1, 1, n)
        theta = (2.0 + 0.13 * 2.0) / 2.0
        want_u = v + (2.0 * np.arange(n) + 1.0) * (rhs - want) / theta
        assert rel(ctx.smooth(0, "chebyshev", 1, v, rhs), want_u) <= TOL_OP
    finally:
        ctx.close()
    if (n, b) == (50, 3):
        g = Golden("band8_1500")
        ctx = Context()
        try:
            ctx.upload_band(1500, 8)
            assert rel(ctx.matvec(0, KIND_A, g["in.L0.v"]), g["out.L0.A_matvec"]) <= TOL_OP
        finally:
            ctx.close()


def test_every_kernel_mapping_gives_the_same_answer(golden_ctx):
    g, ctx = golden_ctx
    o = Oracle(g.hier)
    rng = np.random.default_rng(11)
    try:
        for l, lv in enumerate(g.hier.levels):
            v, b = rng.standard_normal(lv.A.M), rng.standard_normal(lv.A.M)
            want_mv, want_sm = o.matvec(l, KIND_A, v), o.smooth(l, "chebyshev", 2, v, b)
            for m in MAPPINGS:
                ctx.set_mapping(l, KIND_A, m)
                assert rel(ctx.matvec(l, KIND_A, v), want_mv) < TOL_OP, (l, m)
                assert rel(ctx.smooth(l, "chebyshev", 2, v, b), want_sm) < TOL_OP, (l, m)
            if lv.P is not None:
                vc = rng.standard_normal(lv.P.n_local_cols)
                for m in MAPPINGS:
                    ctx.set_mapping(l, KIND_P, m)
                    ctx.set_mapping(l, KIND_R, m)
                    assert rel(ctx.matvec(l, KIND_P, vc), o.matvec(l, KIND_P, vc)) < TOL_OP, (l, m)
                    assert rel(ctx.matvec(l, KIND_R, v), o.matvec(l, KIND_R, v)) < TOL_OP, (l, m)
    finally:
        for l, lv in enumerate(g.hier.levels):
            for k in (KIND_A, KIND_P, KIND_R):
                if k == KIND_A or lv.P is not None:
                    ctx.set_mapping(l, k, 0)


def test_mapping_codes_are_canonical(golden_ctx):
    """set_mapping normalises a requested code to one of the codes get_mapping reports: threads per row rounded down
    to a power of two up to 256, streaming lanes to a power of two up to 32, the two sliced layouts as they are; 0
    gives back the rule's choice"""
    g, ctx = golden_ctx
    kept = [1, 16, 32, 256, -1, -32, 100, 101]
    rounded = {3: 2, 17: 16, 31: 16, 33: 32, 99: 64, 102: 64, 255: 128, 300: 256, -3: -2, -64: -32}
    for l, lv in enumerate(g.hier.levels):
        for k in (KIND_A, KIND_P, KIND_R) if lv.P is not None else (KIND_A,):
            at_upload = ctx.get_mapping(l, k)
            try:
                for m in kept:
                    ctx.set_mapping(l, k, m)
                    assert ctx.get_mapping(l, k) == m, (l, k, m)
                for m, want in rounded.items():
                    ctx.set_mapping(l, k, m)
                    assert ctx.get_mapping(l, k) == want, (l, k, m)
            finally:
                ctx.set_mapping(l, k, 0)
            assert ctx.get_mapping(l, k) == at_upload, (l, k)


def test_other_solvers_and_option_sets_against_oracle(golden_ctx):
    g, ctx = golden_ctx
    o = Oracle(g.hier)
    # jacobi smoother, asymmetric sweeps, iteration cap (the `i == max_iter` exit)
    u_o, it_o, h_o = o.solve_pcg(g.rhs, 3, 1e-14, "jacobi", 2, 1)
    u, it, h = ctx.solve_pcg(g.rhs, 3, 1e-14, "jacobi", 2, 1)
    assert it == it_o == 3
    check_pcg(it, h, u, it_o, h_o, u_o)
    # no pre-smoothing / no post-smoothing
    # (one-sided smoothing makes the preconditioner non-symmetric: CG then amplifies rounding
    #  differences as the residual drops, so the history is compared at 1e-7 here; the north_star's
    #  1e-9 applies to the reference's configuration, checked in the tests above)
    for pre, post in ((0, 2), (2, 0)):
        u_o, it_o, h_o = o.solve_pcg(g.rhs, 50, 1e-8, "chebyshev", pre, post)
        u, it, h = ctx.solve_pcg(g.rhs, 50, 1e-8, "chebyshev", pre, post)
        check_pcg(it, h, u, it_o, h_o, u_o, tol_hist=1e-7)
    # saena_object::solve (stationary V-cycles)
    # (its residual is recomputed as A u - rhs every cycle: near convergence that difference
    #  cancels ~8 digits, so two correct evaluations of ||r|| agree only to eps*||rhs||/||r|| ~ 1e-8)
    u_o, it_o, h_o = o.solve_vcycle(g.rhs, 50, 1e-8)
    u, it, h = ctx.solve_vcycle(g.rhs, 50, 1e-8)
    check_pcg(it, h, u, it_o, h_o, u_o, tol_hist=1e-6)
    # saena_object::solve_smoother (the smoother alone as a stationary iteration; iteration cap exit)
    for kw in (dict(max_iter=12, tol=1e-8, smoother="chebyshev", pre=3, post=3), dict(max_iter=7, tol=1e-8, smoother="jacobi", pre=2, post=0)):
        u_s, it_s, h_s = o.solve_smoother(g.rhs, **kw)
        u_g, it_g, h_g = ctx.solve_smoother(g.rhs, **kw)
        assert it_g == it_s and len(h_g) == len(h_s)
        # (as saena_object::solve above: r = A u - rhs is recomputed every iteration, so near convergence two correct
        #  evaluations of ||r|| agree only to eps * ||rhs|| / ||r||: 1e-9 while the residual is large, 1e-6 on the tail)
        err = np.abs(h_g - h_s) / h_s
        head = h_s > 1e-5 * h_s[0]
        assert err[head].max() <= TOL_HIST and err.max() <= 1e-6 and rel(u_g, u_s) <= 1e-9, err
    # saena_object::solve_CG (unpreconditioned): must converge to the same solution
    u_cg, it_cg, h_cg = ctx.solve_cg(g.rhs, 2000, 1e-10)
    assert h_cg[-1] / h_cg[0] < 1e-10
    assert rel(u_cg, u_o) < 1e-6


def _random_csr(rng, n_rows, n_cols, row_nnz):
    counts = np.minimum(np.asarray(row_nnz, np.int32), n_cols)
    cols = np.concatenate([np.sort(rng.choice(n_cols, c, replace=False)) for c in counts]) if counts.sum() else \
        np.zeros(0, np.int64)
    return counts, cols.astype(np.int32), rng.uniform(-1, 1, counts.sum())


def _two_level(rng, A_counts, A_cols, A_vals, n, nc=40):
    """a syntactically valid 2-level hierarchy around an arbitrary level-0 operator"""
    def op(kind, level, M, N, counts, cols, vals):
        return Operator(kind=kind, level=level, M=M, Mbig=M, Nbig=N, row_offset=0, col_offset=0, n_local_cols=N,
                        nnzPerRow_local=counts, col_local=cols, val_local=vals)
    pc, pcol, pv = _random_csr(rng, n, nc, rng.integers(0, 4, n))
    rc, rcol, rv = _random_csr(rng, nc, n, rng.integers(0, 30, nc))
    dense = rng.uniform(-1, 1, (nc, nc)) + nc * np.eye(nc)
    cr, cc = np.nonzero(dense)
    lv0 = Level(0, op(KIND_A, 0, n, n, A_counts, A_cols, A_vals), inv_diag=rng.uniform(0.5, 1.5, n), eig_max=1.7,
                P=op(KIND_P, 0, n, nc, pc, pcol, pv), R=op(KIND_R, 0, nc, n, rc, rcol, rv), M_coarse_old=nc,
                M_coarse=nc)
    lv1 = Level(1, op(KIND_A, 1, nc, nc, np.full(nc, nc, np.int32), np.tile(np.arange(nc, dtype=np.int32), nc),
                      dense.ravel()), inv_diag=1.0 / np.diag(dense), eig_max=1.5)
    return Hierarchy([lv0, lv1], coarse_n=nc, coarse_row=cr.astype(np.int32), coarse_col=cc.astype(np.int32),
                     coarse_val=dense[cr, cc])


@pytest.mark.parametrize("case", ["ragged", "empty_rows", "one_long_row", "dense_rows", "single_row"])
def test_edge_case_row_shapes(case):
    """ragged rows, empty rows, a row longer than the streaming tile, wide rows -- every mapping"""
    rng = np.random.default_rng(99)
    n = {"single_row": 1}.get(case, 3000)
    if case == "ragged":
        nnz = rng.integers(0, 70, n)
    elif case == "empty_rows":
        nnz = np.where(rng.random(n) < 0.6, 0, rng.integers(1, 9, n))
    elif case == "one_long_row":
        nnz = rng.integers(1, 8, n)
        nnz[[0, 1500, n - 1]] = [2900, 2500, 2100]   # > STREAM_TILE (2048)
    elif case == "dense_rows":
        nnz = np.full(n, 300)
    else:
        nnz = np.array([1])
    counts, cols, vals = _random_csr(rng, n, n, nnz)
    h = _two_level(rng, counts, cols, vals, n)
    o = Oracle(h)
    ctx = Context()
    try:
        ctx.upload_hierarchy(h)
        v, b = rng.standard_normal(n), rng.standard_normal(n)
        want, want_res = o.matvec(0, KIND_A, v), o.residual(0, v, b)
        want_cheb, want_jac = o.smooth(0, "chebyshev", 3, v, b), o.smooth(0, "jacobi", 2, v, b)
        scale = np.linalg.norm(want) or 1.0
        for m in MAPPINGS:
            ctx.set_mapping(0, KIND_A, m)
            assert np.linalg.norm(ctx.matvec(0, KIND_A, v) - want) <= TOL_OP * scale, (case, m)
            assert rel(ctx.residual(0, v, b), want_res) < TOL_OP, (case, m)
            assert rel(ctx.smooth(0, "chebyshev", 3, v, b), want_cheb) < TOL_OP, (case, m)
            assert rel(ctx.smooth(0, "jacobi", 2, v, b), want_jac) < TOL_OP, (case, m)
        vc = rng.standard_normal(40)
        assert rel(ctx.matvec(0, KIND_P, vc), o.matvec(0, KIND_P, vc)) < TOL_OP
        assert rel(ctx.matvec(0, KIND_R, v), o.matvec(0, KIND_R, v)) < TOL_OP
        assert rel(ctx.vcycle(0, v, b), o.vcycle(0, v, b)) < 1e-11
    finally:
        ctx.close()


def test_cuda_graph_replay_is_bitwise_the_eager_solve(golden_ctx):
    g, ctx = golden_ctx
    ctx.set_graphs(False)
    u0, it0, h0 = ctx.solve_pcg(g.rhs, g.max_iter, g.tol)
    ctx.set_graphs(True)
    n0 = ctx.launch_count()
    u1, it1, h1 = ctx.solve_pcg(g.rhs, g.max_iter, g.tol)   # captures on the first V-cycle, replays after
    u2, it2, h2 = ctx.solve_pcg(g.rhs, g.max_iter, g.tol)   # replays only
    assert it0 == it1 == it2
    assert np.array_equal(h0, h1) and np.array_equal(h0, h2)
    assert np.array_equal(u0, u1) and np.array_equal(u0, u2)
    assert ctx.launch_count() > n0


def test_coarsest_cg_option(golden_ctx):
    """direct_solver == "CG": solve_coarsest_CG (saena_object_solve.cpp:14-114) instead of the direct solve"""
    g, ctx = golden_ctx
    o = Oracle(g.hier, coarsest_cg=True)
    ctx.set_coarsest_solver("CG")
    try:
        b = np.random.default_rng(4).standard_normal(g.hier.levels[0].A.M)
        assert rel(ctx.vcycle(0, np.zeros_like(b), b), o.vcycle(0, np.zeros_like(b), b)) < 1e-11
        u_o, it_o, h_o = o.solve_pcg(g.rhs, g.max_iter, g.tol)
        u, it, h = ctx.solve_pcg(g.rhs, g.max_iter, g.tol)
        check_pcg(it, h, u, it_o, h_o, u_o)
    finally:
        ctx.set_coarsest_solver("SuperLU")


def test_scale_hooks():
    """saena_object::scale == true: the V-cycle multiplies the restricted residual and the coarse
    correction by the coarse level's D^-1/2 and the solvers scale the final u
    (saena_object_solve.cpp:1245-1247, :1264-1266, :2709-2711).  Checked against the oracle's
    restatement: the reference itself cannot run this path (see oracle/ref.py)."""
    g = Golden(GOLDEN[1])
    h = g.hier
    rng = np.random.default_rng(8)
    h.scale = True
    for lv in h.levels:
        lv.inv_sq_diag = rng.uniform(0.8, 1.25, lv.A.M)
    o = Oracle(h)
    ctx = Context()
    try:
        ctx.upload_hierarchy(h)
        b = rng.standard_normal(h.levels[0].A.M)
        assert rel(ctx.vcycle(0, np.zeros_like(b), b), o.vcycle(0, np.zeros_like(b), b)) < 1e-11
        u_o, it_o, h_o = o.solve_pcg(g.rhs, 50, 1e-8)
        u, it, hist = ctx.solve_pcg(g.rhs, 50, 1e-8)
        check_pcg(it, hist, u, it_o, h_o, u_o, tol_hist=1e-7)   # scaled V-cycle is not symmetric
        # and it differs from the unscaled solve, i.e. the hooks really ran
        h.scale = False
        u_plain, _, _ = Oracle(h).solve_pcg(g.rhs, 50, 1e-8)
        assert rel(u, u_plain) > 1e-3
    finally:
        ctx.close()


def test_dot_and_linearity_properties():
    g = Golden(GOLDEN[1])
    ctx = Context()
    try:
        ctx.upload_hierarchy(g.hier)
        rng = np.random.default_rng(1)
        n = g.hier.levels[0].A.M
        x, y = rng.standard_normal(n), rng.standard_normal(n)
        a = 0.37
        lin = ctx.matvec(0, KIND_A, a * x + y)
        assert rel(lin, a * ctx.matvec(0, KIND_A, x) + ctx.matvec(0, KIND_A, y)) < 1e-13
        # R = P^T (restrict_matrix.cpp:116-121): <R x, z> == <x, P z>
        z = rng.standard_normal(g.hier.levels[0].P.n_local_cols)
        lhs = float(ctx.matvec(0, KIND_R, x) @ z)
        rhs = float(x @ ctx.matvec(0, KIND_P, z))
        assert abs(lhs - rhs) <= 1e-12 * abs(lhs)
        big = rng.standard_normal(3_000_001)
        assert abs(ctx.dot(big, big) - float(big @ big)) <= 1e-12 * float(big @ big)
        assert ctx.dot(np.zeros(0), np.zeros(0)) == 0.0
    finally:
        ctx.close()


@pytest.mark.ref
@pytest.mark.parametrize("mx", [20, 34])
def test_cuda_vs_compiled_reference_same_process_same_hierarchy(mx):
    """BASELINE.json configs[0] (Poisson 32^3, via experiments/Poisson.cpp's sequence) and a smaller
    one: reference setup on the host, hierarchy uploaded once, then both solve on the same
    hierarchy object in this process."""
    from oracle import ref
    s = ref.RefSolver.poisson(mx)
    ctx = Context()
    try:
        h = s.hierarchy()
        ctx.upload_hierarchy(h)
        rng = np.random.default_rng(2)
        for l, lv in enumerate(h.levels):
            v, b = rng.standard_normal(lv.A.M), rng.standard_normal(lv.A.M)
            assert rel(ctx.matvec(l, KIND_A, v), s.matvec(l, KIND_A, v)) < TOL_OP
            assert rel(ctx.smooth(l, "chebyshev", 3, v, b), s.smooth(l, "chebyshev", 3, v, b)) < TOL_OP
            assert rel(ctx.smooth(l, "jacobi", 1, v, b), s.smooth(l, "jacobi", 1, v, b)) < TOL_OP
            if lv.P is not None:
                vc = rng.standard_normal(lv.P.n_local_cols)
                assert rel(ctx.matvec(l, KIND_P, vc), s.matvec(l, KIND_P, vc)) < TOL_OP
                assert rel(ctx.matvec(l, KIND_R, v), s.matvec(l, KIND_R, v)) < TOL_OP
            assert rel(ctx.vcycle(l, np.zeros(lv.A.M), b), s.vcycle(l, np.zeros(lv.A.M), b)) < 1e-11
        u_ref, it_ref, hist_ref = s.solve_pcg()
        u, it, hist = ctx.solve_pcg(s.rhs(), s.opts.max_iter, s.opts.tol, "chebyshev", s.opts.pre, s.opts.post)
        assert it == it_ref
        check_pcg(it, hist, u, it_ref, hist_ref, u_ref, TOL_HIST)
    finally:
        ctx.close()
        s.close()


def test_fused_residual_restrict_measurement_kernel_matches_the_two_kernels():
    """csrc/fused_restrict.cu (the measurement behind 'restriction fused with the residual'): the scatter form with
    FP64 atomics gives the solve path's res_coarse = R (A u - rhs) within the per-operator tolerance"""
    g = Golden(GOLDEN[1])
    ctx = Context()
    rng = np.random.default_rng(21)
    try:
        ctx.upload_hierarchy(g.hier)
        for l, lv in enumerate(g.hier.levels[:-1]):
            ctx.set_mapping(l, KIND_A, 100)
            u, b = rng.uniform(-1, 1, lv.A.M), rng.uniform(-1, 1, lv.A.M)
            t2, t1, diff = ctx.time_residual_restrict(l, u, b, 3)
            assert diff <= TOL_OP and t1 > 0 and t2 > 0, (l, diff)
            want = Oracle(g.hier).matvec(l, KIND_R, Oracle(g.hier).residual(l, u, b))
            assert rel(ctx.matvec(l, KIND_R, ctx.residual(l, u, b)), want) <= TOL_OP
        # the same form inside the V-cycle of a PCG solve (opt-in): iteration count and history of the oracle
        u_o, it_o, h_o = Oracle(g.hier).solve_pcg(g.rhs, g.max_iter, g.tol, "chebyshev", g.pre, g.post)
        launches = ctx.launch_count()
        ctx.set_fused_restrict(len(g.hier.levels))
        u1, it1, h1 = ctx.solve_pcg(g.rhs, g.max_iter, g.tol, "chebyshev", g.pre, g.post)
        n_fused = ctx.launch_count() - launches
        ctx.set_fused_restrict(0)
        u2, it2, h2 = ctx.solve_pcg(g.rhs, g.max_iter, g.tol, "chebyshev", g.pre, g.post)
        check_pcg(it1, h1, u1, it_o, h_o, u_o)
        check_pcg(it2, h2, u2, it_o, h_o, u_o)
        assert n_fused < ctx.launch_count() - launches - n_fused   # one launch less per level and V-cycle
    finally:
        ctx.close()
