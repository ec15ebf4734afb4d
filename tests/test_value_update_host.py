"""The host reference of saena_b200_update_values (tests/value_update_ref.py) pinned to the setup: with the values the
hierarchy was built from, R A P mapped onto each stored pattern by the lumping rule reproduces every stored coarse
operator, its inv_diag and the coarsest COO -- the rule is the setup's filter, not only the tests' idea of it."""
import numpy as np
import pytest

from saena_b200.sa_setup import build_hierarchy, poisson3d_coo, unstructured2d_coo
from tests.value_update_ref import map_onto_pattern, rescaled_values, shifted_values, updated_hierarchy


def _rel_max(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / np.max(np.abs(np.asarray(b))))


@pytest.fixture(scope="module", params=["poisson24", "unstructured40"])
def hier(request):
    if request.param == "poisson24":
        return build_hierarchy(*poisson3d_coo(24), device="cpu")
    return build_hierarchy(*unstructured2d_coo(40), device="cpu")


def test_unchanged_values_reproduce_every_stored_level(hier):
    assert len(hier.levels) >= 3
    h, fracs = updated_hierarchy(hier, hier.levels[0].A.val_local)
    assert len(fracs) == len(hier.levels) and fracs[0] == 0.0
    for new, old in zip(h.levels, hier.levels):
        assert np.array_equal(new.A.col_local, old.A.col_local)
        assert _rel_max(new.A.val_local, old.A.val_local) < 1e-13, new.level
        assert _rel_max(new.inv_diag, old.inv_diag) < 1e-13, new.level
    assert np.array_equal(h.coarse_row, hier.coarse_row) and np.array_equal(h.coarse_col, hier.coarse_col)
    assert _rel_max(h.coarse_val, hier.coarse_val) < 1e-13
    # the setup filtered small entries from the deeper products: the fractions are small, not all zero
    assert all(0.0 <= f < 1e-6 for f in fracs)


def test_new_values_keep_patterns_and_report_lumped_mass(hier):
    A0 = hier.levels[0].A
    for vals in (shifted_values(A0, 0.5), rescaled_values(A0, 1.0 + 0.5 * np.sin(np.arange(A0.M) * 0.37))):
        h, fracs = updated_hierarchy(hier, vals)
        for new, old in zip(h.levels, hier.levels):
            assert np.array_equal(new.A.nnzPerRow_local, old.A.nnzPerRow_local)
            assert np.all(np.isfinite(new.A.val_local)) and np.all(np.isfinite(new.inv_diag))
        assert fracs[0] == 0.0 and all(0.0 <= f < 1.0 for f in fracs)
        # a new value set changes the coarse operators
        assert _rel_max(h.levels[1].A.val_local, hier.levels[1].A.val_local) > 1e-6


def test_stored_entry_missing_from_the_product_is_an_error(hier):
    import scipy.sparse as sp
    op = hier.levels[1].A
    C = sp.csr_matrix((np.ones(op.M), (np.arange(op.M), np.arange(op.M))), shape=(op.M, op.M))   # diagonal only
    with pytest.raises(ValueError, match="not a Galerkin product"):
        map_onto_pattern(C, op)
