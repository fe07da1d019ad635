"""Pins the CPU oracle against what the UNMODIFIED reference modules return for the same seeded inputs
(tests/golden/oracle_reference.npz and the ``grid6_hex`` graph of tests/golden/graphs.npz, both generated from the running
reference: tests/golden/make_golden_oracle.py, tests/golden/make_golden_graphs.py)."""

from __future__ import annotations

import os

import numpy as np
import pytest

from oracle import ref
from tests.golden.make_golden_oracle import NHOOD_CASES, NHOOD_PERMS, NHOOD_SEED, cooc_case, interaction_cases, nhood_case
from tools import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(os.path.join(GOLDEN, "oracle_reference.npz"), allow_pickle=False))


def test_hex_graph_matches_gridbuilder():
    gold = np.load(os.path.join(GOLDEN, "graphs.npz"), allow_pickle=False)  # GridBuilder(n_neighs=6) on hex_coords(23, 31)
    g = synth.hex_graph(23, 31)
    np.testing.assert_array_equal(g.indptr, gold["grid6_hex_adj_indptr"])
    np.testing.assert_array_equal(g.indices, gold["grid6_hex_adj_indices"])
    np.testing.assert_array_equal(g.data, gold["grid6_hex_adj_data"])
    assert g.dtype == np.float32 and g.indices.dtype == np.int32


@pytest.mark.parametrize("n_cls,libs", NHOOD_CASES)
def test_nhood_perms_vs_reference(gold, n_cls, libs):
    ptr, ind, lab, libraries = nhood_case(n_cls, libs)
    np.testing.assert_array_equal(ref.nhood_count(ptr, ind, lab, n_cls), gold[f"nhood{n_cls}_count"])
    got = ref.nhood_perm_counts(ptr, ind, lab, n_cls, ref.spawn_states(NHOOD_SEED, NHOOD_PERMS),
                                None if libraries is None else libraries.cat.codes.to_numpy(), 3 if libs else 0)
    np.testing.assert_array_equal(got, gold[f"nhood{n_cls}_perms"])


def test_cooc_vs_reference(gold):
    pts, lb, iv = cooc_case()
    np.testing.assert_array_equal(ref.occur_count(pts[:, 0], pts[:, 1], iv[1:] ** 2, lb, 5), gold["cooc_counts"])
    occ, _ = ref.co_occurrence_helper(pts[:, 0], pts[:, 1], iv, lb)
    np.testing.assert_allclose(occ, gold["cooc_occ"], rtol=1e-12)


def test_pair_counts_vs_sklearn():
    from sklearn.neighbors import KDTree

    rr = np.random.default_rng(9)
    P = rr.random((2500, 2)) * 100
    sup = np.linspace(0, 70, 50)
    np.testing.assert_array_equal(ref.pair_counts(P, sup), KDTree(P).two_point_correlation(P, sup, dualtree=True))


def test_interaction_matrix_oracle_kat_and_reference(gold):
    """Oracle restatement of interaction_matrix (next row of SURVEY 8f): the reference's own known answers
    (tests/graph/test_nhood.py:153-173, fixture tests/conftest.py:177-194) and its numba kernel on random graphs."""
    import scipy.sparse as sp

    g = sp.csr_matrix(np.array([[0, 1, 1, 0, 0], [0, 0, 0, 0, 1], [1, 2, 0, 0, 0], [0, 1, 0, 0, 1], [0, 0, 1, 2, 0]]))
    codes = np.array([0, 0, 0, 1, 1])
    np.testing.assert_array_equal(ref.interaction_matrix(g, codes, 2, weights=True), [[5, 1], [2, 3]])
    np.testing.assert_array_equal(ref.interaction_matrix(g, codes, 2, weights=False), [[4, 1], [2, 2]])
    nan_codes = np.array([-1, 0, 0, 1, 1])
    np.testing.assert_array_equal(ref.interaction_matrix(g, nan_codes, 2, weights=True), [[2, 1], [2, 3]])
    np.testing.assert_array_equal(ref.interaction_matrix(g, nan_codes, 2, weights=False), [[1, 1], [2, 2]])
    assert ref.interaction_matrix(g, codes, 2).dtype == np.int64
    np.testing.assert_allclose(ref.interaction_matrix(g, codes, 2, normalized=True).sum(1), 1.0)

    for name, a, codes, k in interaction_cases():
        for weights in (False, True):
            got = ref.interaction_matrix(a, codes, k, weights=weights)
            assert got.dtype == np.float64
            np.testing.assert_array_equal(got, gold[f"interaction_{name}_w{int(weights)}"])  # same accumulation order: bit-identical float sums
