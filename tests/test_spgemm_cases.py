"""The dispatch of the device SpGEMM as restated in tests/spgemm_cases.py, and the coverage each case there claims, at
a B200's constants (148 SMs, 232 448 bytes of opt-in shared memory per block).  No GPU needed: a change to a case or
to the dispatch that loses a kernel path, a bin edge or a CTA's second row fails here."""
import dataclasses

import numpy as np
import pytest

from tests import spgemm_cases as sc

SMS, SMEM = sc.B200_SMS, sc.B200_SMEM_OPTIN


def test_dispatch_limits_at_b200_constants():
    # worked out by hand from spgemm.cu: the shared bitmask holds n_words * 4 + 64 <= 232 448 bytes, the shared dense
    # accumulator (N + ceil(n_words / 2)) * 8 + 2048 <= 232 448 bytes
    assert sc.symbolic_limits(1_859_072, SMEM)[5] == 1_859_072
    assert sc.symbolic_limits(1_859_073, SMEM)[5] == 8192
    assert not sc.numeric_dense_slab(28_356, SMEM) and sc.numeric_dense_slab(28_357, SMEM)
    assert sc.numeric_limits(20_000, SMEM) == (0, 32, 128, 512, 4096, 8192, 20_000)
    many = 10 ** 6
    assert sc.grid("symbolic", 5, many, 20_000, SMS, SMEM) == 8 * 148
    assert sc.grid("symbolic", 6, many, 2_000_000, SMS, SMEM) == 4 * 148
    assert sc.grid("numeric", 6, many, 20_000, SMS, SMEM) == 148
    assert sc.grid("numeric", 6, many, 2_000_000, SMS, SMEM) == 132        # 2 GiB / 16.25 MB
    assert [sc.scan_blocks(m) for m in (0, 1, 1024, 1025, 3_000_017)] == [1, 1, 1, 2, 2930]


def test_bins_at_their_edges():
    sizes = [0, 1, 32, 33, 128, 129, 512, 513, 4096, 4097, 8192, 8193, 10 ** 6]
    assert list(sc.symbolic_bin(sizes, 20_000, SMEM)) == [0, 1, 1, 2, 2, 3, 3, 4, 4, 4, 4, 5, 5]
    assert list(sc.symbolic_bin(sizes, 2_000_000, SMEM)) == [0, 1, 1, 2, 2, 3, 3, 4, 4, 4, 4, 6, 6]
    assert list(sc.numeric_bin(sizes[:-1], 20_000, SMEM)) == [0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6]
    assert list(sc.symbolic_bin([10_000, 40, 33], 40, SMEM)) == [2, 2, 2]    # capped at N = 40


def test_hash_restatement_puts_the_expected_columns_on_each_last_slot():
    every = np.arange(2_000_000)
    counts = [int((sc.sg_hash(every, t - 1) == t - 1).sum()) for t in (64, 256, 1024, 8192, 16384)]
    assert counts == [31_251, 7_812, 1_953, 244, 122]


@pytest.mark.parametrize("name", sc.NAMES)
def test_case_covers_what_it_claims_on_a_b200(name):
    case = sc.build(name)
    assert case.claims
    assert sc.unmet_claims(case, SMS, SMEM) == []
    # every case is checked bit for bit on the GPU: its sums must be exact in any order
    assert sc.values_are_exact(case.A, case.B, sc.structure(case.A, case.B).data)


@pytest.mark.parametrize("name,launch", [("bitmask_shared_reused", "symbolic"), ("dense_shared_reused", "numeric"),
                                         ("global_bitmask_and_slab_reused", "symbolic")])
def test_reuse_claims_fail_on_a_card_with_more_ctas_than_rows(name, launch):
    """the claim of a CTA's second row is a real condition: with ten times the SMs the grid covers the bin (the global
    dense slab's grid is bounded by its 2 GiB budget, not by the SMs)"""
    unmet = sc.unmet_claims(sc.build(name), 10 * SMS, SMEM)
    assert len(unmet) == 1 and f"Rows(pass_='{launch}'" in unmet[0]


def test_claims_fail_where_the_case_does_not_reach():
    case = sc.build("probe_wraparound")
    shifted = [dataclasses.replace(c, at_least=c.at_least + 1) for c in case.claims]
    assert len(sc.unmet_claims(dataclasses.replace(case, claims=tuple(shifted)), SMS, SMEM)) == len(shifted)
    case = sc.build("structural_zeros")
    assert sc.unmet_claims(dataclasses.replace(case, claims=(sc.Zeros(0, 1),)), SMS, SMEM)
