"""Level route (saena_b200_set_level_route, csrc/solve.cu:sb_apply_level_A): level 1's operator applied as
R_0 (A_0 (P_0 x)) instead of streaming the stored Galerkin product.  On the 64^3 Poisson device hierarchy the route
must give the stored operator's results to rounding -- matvec (also against scipy on the host), the smoother sweeps,
the residual, a V-cycle, the PCG solve -- replay bitwise from a CUDA graph, report the three operators' bytes, and be
refused where the stored A_1 is not R_0 A_0 P_0."""
import copy
import dataclasses

import numpy as np
import pytest


def _cuda() -> bool:
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _cuda(), reason="needs a CUDA device")]

N = 64
TOL = 1e-12


def rel(a, b):
    return float(np.linalg.norm(np.asarray(a) - np.asarray(b)) / np.linalg.norm(np.asarray(b)))


@pytest.fixture(scope="module")
def hier():
    from saena_b200 import sa_setup
    dh = sa_setup.build_device_hierarchy(*sa_setup.poisson3d_coo(N), device="cuda")
    h = dh.to_rank(0, 1)
    del dh
    import torch
    torch.cuda.empty_cache()
    assert len(h.levels) >= 3
    return h


@pytest.fixture()
def ctx(hier):
    from saena_b200.native import Context
    c = Context()
    c.upload_hierarchy(hier)
    yield c
    c.close()


def test_route_matvec_and_bytes(ctx, hier):
    from saena_b200.hierarchy import KIND_A, KIND_P, KIND_R
    x = np.random.default_rng(1).uniform(-1, 1, hier.levels[1].A.M)
    stored = ctx.matvec(1, KIND_A, x)
    stored_bytes = ctx.operator_bytes(1, KIND_A)
    assert not ctx.get_level_route(1)
    ctx.set_level_route(1, True)
    assert ctx.get_level_route(1)
    route = ctx.matvec(1, KIND_A, x)
    assert rel(route, stored) <= TOL
    assert rel(route, hier.levels[1].A.to_scipy_local() @ x) <= TOL
    assert ctx.operator_bytes(1, KIND_A) == sum(ctx.operator_bytes(0, k) for k in (KIND_A, KIND_P, KIND_R))
    assert ctx.operator_bytes(1, KIND_A) < stored_bytes
    assert ctx.time_matvec(1, KIND_A, 3) > 0.0
    ctx.set_level_route(1, False)
    assert not ctx.get_level_route(1)
    assert ctx.operator_bytes(1, KIND_A) == stored_bytes
    assert np.array_equal(ctx.matvec(1, KIND_A, x), stored)


def test_route_sweeps_residual_vcycle(ctx, hier):
    M = hier.levels[1].A.M
    rng = np.random.default_rng(2)
    u, rhs = rng.uniform(-1, 1, M), rng.uniform(-1, 1, M)

    def run():
        return {"cheb1": ctx.smooth(1, "chebyshev", 1, u, rhs),      # Chebyshev first sweep
                "cheb3": ctx.smooth(1, "chebyshev", 3, u, rhs),      # ... and the following ones
                "jacobi": ctx.smooth(1, "jacobi", 2, u, rhs),
                "residual": ctx.residual(1, u, rhs),
                "vcycle": ctx.vcycle(1, u, rhs)}

    stored = run()
    ctx.set_level_route(1, True)
    route = run()
    for k in stored:
        assert rel(route[k], stored[k]) <= TOL, k


def test_route_pcg_and_graph_replay(ctx, hier):
    from saena_b200.sa_setup import poisson3d_rhs
    rhs = poisson3d_rhs(N)
    _, it0, h0 = ctx.solve_pcg(rhs)
    ctx.set_level_route(1, True)
    u1, it1, h1 = ctx.solve_pcg(rhs)            # captured into a new graph (set_level_route dropped the old one)
    replays = ctx.graph_replays()
    u2, it2, h2 = ctx.solve_pcg(rhs)            # replayed
    assert ctx.graph_replays() > replays
    assert it1 == it0 and np.all(np.abs(h1 - h0) <= 1e-9 * np.abs(h0))
    ctx.set_graphs(False)
    u3, it3, h3 = ctx.solve_pcg(rhs)            # eager
    ctx.set_graphs(True)
    assert it2 == it3 == it1
    assert np.array_equal(u2, u3) and np.array_equal(h2, h3) and np.array_equal(u1, u2)


def test_route_refused_where_not_allowed(ctx):
    from saena_b200.native import NativeError
    with pytest.raises(NativeError, match="no level above"):
        ctx.set_level_route(0, True)
    assert not ctx.get_level_route(0)
    assert ctx.get_level_route(99) is False


def test_autotune_takes_the_route_where_it_measures_faster(ctx, hier):
    """saena_b200_autotune_mapping's route rule, level by level: a level is timed both ways exactly when the three
    operators of the level above stream fewer bytes than its stored A (the coarsest level never), and it takes the
    route exactly when the route's sweep beat the stored one by more than min_gain"""
    from saena_b200.hierarchy import KIND_A, KIND_P, KIND_R
    L = len(hier.levels)
    stored = [ctx.operator_bytes(l, KIND_A) for l in range(L)]
    three = [sum(ctx.operator_bytes(l, k) for k in (KIND_A, KIND_P, KIND_R)) for l in range(L - 1)]
    assert three[0] < stored[1]               # 64^3 Poisson: the route is worth timing on level 1
    for min_gain in (0.03, 0.99):
        ctx.autotune_mapping_native(10, min_gain)
        for l in range(L):
            on, ms_stored, ms_route = ctx.level_route_choice(l)
            timed = 1 <= l < L - 1 and three[l - 1] < stored[l]
            assert (ms_stored > 0 and ms_route > 0) == timed, l
            assert on == (timed and ms_route < (1 - min_gain) * ms_stored), (l, min_gain, ms_stored, ms_route)
            assert ctx.operator_bytes(l, KIND_A) == (three[l - 1] if on else stored[l])
    assert not any(ctx.get_level_route(l) for l in range(L))   # nothing is 100x faster


def test_probe_refuses_an_operator_that_is_not_rap(hier):
    """A_1 scaled by (1 + 1e-6) before upload: forcing the route fails the probe check, and the autotuner keeps the
    stored operator (the solve must use the uploaded A_1, whatever it is)"""
    from saena_b200.hierarchy import KIND_A
    from saena_b200.native import Context, NativeError
    h = copy.copy(hier)
    h.levels = list(hier.levels)
    lv1 = hier.levels[1]
    h.levels[1] = dataclasses.replace(lv1, A=dataclasses.replace(lv1.A, val_local=lv1.A.val_local * (1 + 1e-6)))
    c = Context()
    try:
        c.upload_hierarchy(h)
        with pytest.raises(NativeError, match="differs from the stored operator"):
            c.set_level_route(1, True)
        assert not c.get_level_route(1)
        c.autotune_mapping_native(3, 0.0)
        assert not c.get_level_route(1)
        x = np.random.default_rng(3).uniform(-1, 1, lv1.A.M)
        assert rel(c.matvec(1, KIND_A, x), h.levels[1].A.to_scipy_local() @ x) <= TOL
    finally:
        c.close()
