"""saena_b200_update_values (csrc/refresh.cu): new values for level 0's operator, every coarse level recomputed as
R A P on its stored pattern.  On the 64^3 Poisson device hierarchy (and the unstructured shape) the updated context must
apply the operators, diagonals and Chebyshev bounds of a fresh context holding the host reference's hierarchy
(tests/value_update_ref.py), solve like it, keep forced mappings and their layouts right, keep or drop the level route
by its probe, refuse what it cannot do without touching the hierarchy, and un-finalize itself on a failure mid-way."""
import copy

import numpy as np
import pytest


def _cuda() -> bool:
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _cuda(), reason="needs a CUDA device")]

SEED = 7
KIND_A = 0


def rel(a, b):
    return float(np.linalg.norm(np.asarray(a) - np.asarray(b)) / np.linalg.norm(np.asarray(b)))


def hist_close(a, b, tol=1e-9):
    a, b = np.asarray(a), np.asarray(b)
    return len(a) == len(b) and float(np.max(np.abs(a - b) / np.abs(b))) < tol


def _device_hier(shape):
    from saena_b200 import sa_setup
    import torch
    coo = sa_setup.poisson3d_coo(64) if shape == "poisson64" else sa_setup.unstructured2d_coo(160)
    dh = sa_setup.build_device_hierarchy(*coo, device="cuda")
    h = dh.to_rank(0, 1)
    del dh
    torch.cuda.empty_cache()
    assert len(h.levels) >= 3 if shape == "poisson64" else len(h.levels) >= 2
    return h


@pytest.fixture(scope="module")
def poisson():
    return _device_hier("poisson64")


@pytest.fixture(scope="module")
def unstructured():
    return _device_hier("unstructured")


def _ctx(h):
    from saena_b200.native import Context
    c = Context()
    c.upload_hierarchy(h)
    return c


def _value_sets(h):
    from tests.value_update_ref import rescaled_values, shifted_values
    A0 = h.levels[0].A
    row = np.repeat(np.arange(A0.M), A0.nnzPerRow_local)
    sigma = 0.2 * float(np.mean(np.abs(A0.val_local[row == np.asarray(A0.col_local)])))   # a fifth of the diagonal
    d = 1.0 + 0.5 * np.sin(np.arange(A0.M) * 0.013)
    return {"shift": shifted_values(A0, sigma), "dad": rescaled_values(A0, d)}


def _csr(op):
    from tests.value_update_ref import _csr
    return _csr(op)


def _snapshot(ctx, h):
    rng = np.random.default_rng(3)
    return [ctx.matvec(l, KIND_A, rng.uniform(-1, 1, lv.A.M)) for l, lv in enumerate(h.levels)]


def _rhs(h):
    return np.random.default_rng(11).uniform(-1, 1, h.levels[0].A.M)


@pytest.mark.parametrize("shape", ["poisson64", "unstructured"])
@pytest.mark.parametrize("which", ["shift", "dad"])
def test_update_matches_a_context_holding_the_reference_hierarchy(shape, which, request):
    from tests.value_update_ref import updated_hierarchy
    h = request.getfixturevalue("poisson" if shape == "poisson64" else "unstructured")
    vals = _value_sets(h)[which]
    href, fracs_ref = updated_hierarchy(h, vals)
    live, ref = _ctx(h), _ctx(href)
    try:
        rhs = _rhs(h)
        live.solve_pcg(rhs)                          # captures a V-cycle with the old constants
        for l in range(len(h.levels)):
            ref.find_eig(l, 20, seed=SEED, store=True)
        fracs = live.update_values(vals, 20, SEED)
        assert len(fracs) == len(h.levels) and fracs[0] == 0.0
        assert np.allclose(fracs, fracs_ref, rtol=0, atol=1e-10)
        rng = np.random.default_rng(5)
        for l, lv in enumerate(href.levels):
            x, b = rng.uniform(-1, 1, lv.A.M), rng.uniform(-1, 1, lv.A.M)
            w = live.matvec(l, KIND_A, x)
            assert rel(w, ref.matvec(l, KIND_A, x)) < 1e-12, l
            assert rel(w, _csr(lv.A) @ x) < 1e-12, l
            assert rel(live.residual(l, x, b), ref.residual(l, x, b)) < 1e-12, l
            # Jacobi reads inv_diag, Chebyshev reads eig_max as well
            assert rel(live.smooth(l, "jacobi", 2, x, b), ref.smooth(l, "jacobi", 2, x, b)) < 1e-12, l
            assert rel(live.smooth(l, "chebyshev", 2, x, b), ref.smooth(l, "chebyshev", 2, x, b)) < 1e-10, l
        u1, it1, h1 = live.solve_pcg(rhs)
        u2, it2, h2 = live.solve_pcg(rhs)
        live.set_graphs(False)
        u3, it3, h3 = live.solve_pcg(rhs)
        assert np.array_equal(u1, u2) and np.array_equal(u1, u3) and np.array_equal(h1, h3)
        ur, itr, hr = ref.solve_pcg(rhs)
        assert it1 == itr and hist_close(h1, hr)
    finally:
        live.close()
        ref.close()


def test_identity_update_changes_nothing(poisson):
    h = poisson
    ctx = _ctx(h)
    try:
        for l in range(len(h.levels)):
            ctx.find_eig(l, 20, seed=SEED, store=True)
        rhs = _rhs(h)
        before = _snapshot(ctx, h)
        rng = np.random.default_rng(9)
        xs = [(rng.uniform(-1, 1, lv.A.M), rng.uniform(-1, 1, lv.A.M)) for lv in h.levels]
        cheb = [ctx.smooth(l, "chebyshev", 2, x, b) for l, (x, b) in enumerate(xs)]
        _, it0, h0 = ctx.solve_pcg(rhs)
        ctx.update_values(h.levels[0].A.val_local, 20, SEED)
        for a, b in zip(_snapshot(ctx, h), before):
            assert rel(a, b) < 1e-13
        for l, (x, b) in enumerate(xs):
            assert rel(ctx.smooth(l, "chebyshev", 2, x, b), cheb[l]) < 1e-10, l
        _, it1, h1 = ctx.solve_pcg(rhs)
        assert it1 == it0 and hist_close(h1, h0)
    finally:
        ctx.close()


@pytest.mark.parametrize("maps", [(100, 101), (-4, 4)])
def test_forced_mappings_and_their_layouts_follow_the_update(poisson, maps):
    from tests.value_update_ref import updated_hierarchy
    h = poisson
    vals = _value_sets(h)["dad"]
    href, _ = updated_hierarchy(h, vals)
    ctx = _ctx(h)
    try:
        for l, m in enumerate(maps):
            ctx.set_mapping(l, KIND_A, m)
            assert ctx.get_mapping(l, KIND_A) == m
        ctx.update_values(vals, 20, SEED)
        rng = np.random.default_rng(2)
        for l, m in enumerate(maps):
            assert ctx.get_mapping(l, KIND_A) == m
            x = rng.uniform(-1, 1, h.levels[l].A.M)
            assert rel(ctx.matvec(l, KIND_A, x), _csr(href.levels[l].A) @ x) < 1e-12, (l, m)
    finally:
        ctx.close()


@pytest.mark.parametrize("which", ["identity", "shift"])
def test_route_is_kept_only_where_its_probe_passes(poisson, which):
    from tests.value_update_ref import updated_hierarchy
    h = poisson
    vals = h.levels[0].A.val_local if which == "identity" else _value_sets(h)["shift"]
    href, _ = updated_hierarchy(h, vals)
    ctx = _ctx(h)
    try:
        ctx.set_level_route(1, True)
        ctx.update_values(vals, 20, SEED)
        x = np.random.default_rng(4).uniform(-1, 1, h.levels[1].A.M)
        stored = _csr(href.levels[1].A) @ x
        if which == "identity":
            assert ctx.get_level_route(1)
        if ctx.get_level_route(1):
            assert rel(ctx.matvec(1, KIND_A, x), stored) < 1e-11
        else:
            assert rel(ctx.matvec(1, KIND_A, x), stored) < 1e-12   # the stored operator again
    finally:
        ctx.close()


def _refused(ctx, h, vals, match):
    from saena_b200.native import NativeError
    before = _snapshot(ctx, h)
    with pytest.raises(NativeError, match=match):
        ctx.update_values(vals)
    for a, b in zip(_snapshot(ctx, h), before):
        assert np.array_equal(a, b)


def test_refusals_leave_the_hierarchy_untouched(poisson):
    h = poisson
    vals = np.array(h.levels[0].A.val_local, copy=True)
    ctx = _ctx(h)
    try:
        _refused(ctx, h, vals[:-1], "nnz_local")
        A0 = h.levels[0].A
        row = np.repeat(np.arange(A0.M), A0.nnzPerRow_local)
        zero = vals.copy()
        zero[np.flatnonzero(row == np.asarray(A0.col_local))[5]] = 0.0
        _refused(ctx, h, zero, "zero diagonal")
    finally:
        ctx.close()


def test_refusal_on_a_rank_share_of_two():
    from saena_b200 import sa_setup
    from saena_b200.native import Context, NativeError
    h2 = sa_setup.build_device_hierarchy(*sa_setup.poisson3d_coo(16), device="cuda").to_rank(0, 2)
    ctx = Context(rank=0, nranks=2, detached=True)
    try:
        ctx.upload_hierarchy(h2)
        with pytest.raises(NativeError, match="one rank only"):
            ctx.update_values(h2.levels[0].A.val_local)
    finally:
        ctx.close()


def test_refusal_on_a_scaled_hierarchy():
    from saena_b200 import sa_setup
    h = sa_setup.build_device_hierarchy(*sa_setup.poisson3d_coo(16), device="cuda").to_rank(0, 1)
    h = copy.deepcopy(h)
    h.scale = True
    for lv in h.levels:
        lv.inv_sq_diag = np.sqrt(np.abs(lv.inv_diag))
    ctx = _ctx(h)
    try:
        _refused(ctx, h, h.levels[0].A.val_local, "scaled")
    finally:
        ctx.close()


def test_refusal_on_a_sliced_only_operator():
    from saena_b200.native import Context, NativeError
    ctx = Context()
    try:
        nnz = ctx.upload_band(4096, 3, sliced_only=True)
        x = np.random.default_rng(1).uniform(-1, 1, 4096)
        w = ctx.matvec(0, KIND_A, x)
        with pytest.raises(NativeError, match="sliced_only"):
            ctx.update_values(np.ones(nnz))
        assert np.array_equal(ctx.matvec(0, KIND_A, x), w)
    finally:
        ctx.close()


def test_failure_mid_way_unfinalizes_the_context(poisson):
    from saena_b200.native import NativeError
    h = copy.deepcopy(poisson)
    A1 = h.levels[1].A
    # row 0 of A_1 couples to the last coarse row: R_0 A_0 P_0 cannot produce that entry
    n0 = int(A1.nnzPerRow_local[0])
    assert A1.col_local[n0 - 1] < A1.M - 1
    A1.col_local = np.insert(np.asarray(A1.col_local), n0, A1.M - 1).astype(np.int32)
    A1.val_local = np.insert(np.asarray(A1.val_local), n0, -1e-3)
    A1.nnzPerRow_local = np.array(A1.nnzPerRow_local, copy=True)
    A1.nnzPerRow_local[0] += 1
    ctx = _ctx(h)
    try:
        rhs = _rhs(h)
        ctx.solve_pcg(rhs)
        with pytest.raises(NativeError, match="not a Galerkin product"):
            ctx.update_values(h.levels[0].A.val_local)
        with pytest.raises(NativeError, match="finalize"):
            ctx.solve_pcg(rhs)
    finally:
        ctx.close()


def test_device_tensor_gives_the_numpy_result(poisson):
    import torch
    h = poisson
    vals = _value_sets(h)["shift"]
    a, b = _ctx(h), _ctx(h)
    try:
        fa = a.update_values(vals, 20, SEED)
        fb = b.update_values(torch.as_tensor(vals, device="cuda"), 20, SEED)
        assert np.allclose(fa, fb, rtol=0, atol=1e-13)
        for x, y in zip(_snapshot(a, h), _snapshot(b, h)):
            assert rel(x, y) < 1e-13
    finally:
        a.close()
        b.close()
