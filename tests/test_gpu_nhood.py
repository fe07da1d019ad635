"""GPU parity tests for nhood_enrichment (through the C ABI): bit-exact integer counts and numpy-identical shuffles."""

from __future__ import annotations

import numpy as np
import pandas as pd
import pytest
import scipy.sparse as sp

import squidpy_b200 as sq
from oracle import ref
from squidpy_b200._rng import spawn_states
from squidpy_b200.gr import NhoodPlan
from tools import synth

pytestmark = pytest.mark.gpu


def _plan(g, n_cls):
    return NhoodPlan(g.indptr, g.indices, n_cls)


def test_kat1_count():
    plan = NhoodPlan(np.array([0, 2, 3, 5, 7, 9]), np.array([1, 2, 4, 0, 1, 1, 4, 2, 3]), 2)
    out = plan.count(np.array([0, 0, 0, 1, 1]))
    assert out.dtype == np.uint32
    np.testing.assert_array_equal(out, [[4, 1], [2, 2]])


@pytest.mark.parametrize("n_cls", [2, 3, 10, 30, 45, 70, 120, 230, 300])
@pytest.mark.parametrize("single", [1, 0])
def test_count_vs_oracle(n_cls, single):
    # batched path (single=0): n_cls sweeps every histogram layout: 32/16/8/2 permutations per CTA in shared memory, global
    # atomics (230), uint16 labels (300); single=1: the dedicated observed-count kernel (shared histogram up to C=202, else global)
    g = synth.hex_graph(61, 53)
    lab = np.random.default_rng(n_cls).integers(0, n_cls, g.shape[0]).astype(np.uint32)
    plan = _plan(g, n_cls)
    plan.set_option("count_single", single)
    np.testing.assert_array_equal(plan.count(lab), ref.nhood_count(g.indptr, g.indices, lab, n_cls))


def test_count_directed_selfloops_empty_rows():
    rng = np.random.default_rng(0)
    n = 3001
    a = sp.random(n, n, density=0.002, format="csr", random_state=1, dtype=np.float32)
    a = (a + sp.diags((rng.random(n) < 0.3).astype(np.float32), format="csr")).tocsr()
    a.eliminate_zeros()
    a.sort_indices()
    assert (np.diff(a.indptr) == 0).any() and a.diagonal().sum() > 0 and (a != a.T).nnz > 0
    lab = rng.integers(0, 7, n).astype(np.uint32)
    np.testing.assert_array_equal(_plan(a, 7).count(lab), ref.nhood_count(a.indptr, a.indices, lab, 7))
    empty = sp.csr_matrix((5, 5), dtype=np.float32)
    np.testing.assert_array_equal(_plan(empty, 2).count(np.array([0, 1, 0, 1, 1])), np.zeros((2, 2), np.uint32))


@pytest.mark.parametrize("kind", ["hex", "sym_selfloops_unsorted", "knn_directed", "duplicates", "one_missing_mirror", "long_rows"])
def test_count_symmetric_shortcut(kind):
    """Symmetric graphs are counted from the entries with j >= i (each unordered pair once, mirrored increment); anything
    that is not a simple symmetric structure keeps the full CSR.  Both must equal the oracle, observed and permuted."""
    rng = np.random.default_rng(5)
    if kind == "hex":
        g = synth.hex_graph(47, 39)
    elif kind == "sym_selfloops_unsorted":
        a = sp.random(2500, 2500, density=0.003, format="csr", random_state=2, dtype=np.float32)
        g = ((a + a.T) > 0).astype(np.float32) + sp.diags((rng.random(2500) < 0.4).astype(np.float32))
        g = g.tocsr()
        g.eliminate_zeros()
        for i in range(g.shape[0]):  # unsorted column order inside the rows
            b, e = g.indptr[i], g.indptr[i + 1]
            g.indices[b:e] = rng.permutation(g.indices[b:e])
    elif kind == "knn_directed":
        g = synth.knn_graph(rng.random((3000, 2)), 6)
    elif kind == "duplicates":
        base = synth.hex_graph(20, 20).tocoo()
        row, col = np.concatenate([base.row, base.row[:50]]), np.concatenate([base.col, base.col[:50]])
        order = np.argsort(row, kind="stable")
        indptr = np.concatenate([[0], np.cumsum(np.bincount(row, minlength=400))])
        g = sp.csr_matrix((np.ones(row.size, np.float32), col[order].astype(np.int32), indptr.astype(np.int32)), shape=(400, 400))
    elif kind == "one_missing_mirror":
        g = synth.hex_graph(30, 30).tolil()
        g[17, 18] = 0
        g = g.tocsr()
        g.eliminate_zeros()
    else:  # symmetric, but rows longer than the 64 entries the check accepts
        a = sp.random(600, 600, density=0.2, format="csr", random_state=3, dtype=np.float32)
        g = ((a + a.T) > 0).astype(np.float32).tocsr()
    n = g.shape[0]
    n_cls = 11
    lab = rng.integers(0, n_cls, n).astype(np.uint32)
    exp = ref.nhood_count(g.indptr, g.indices, lab, n_cls)
    st = spawn_states(3, 40)
    exp_perm = ref.nhood_perm_counts(g.indptr, g.indices, lab, n_cls, st)
    for count_sym in (-1, 0):
        plan = _plan(g, n_cls)
        plan.set_option("count_sym", count_sym)
        np.testing.assert_array_equal(plan.count(lab), exp)  # dedicated single-vector kernel
        plan.set_option("count_single", 0)                    # the batched kernels, which the shortcut belongs to
        np.testing.assert_array_equal(plan.count(lab), exp)
        plan.set_base(lab)
        np.testing.assert_array_equal(plan.permute(st), exp_perm)


def test_create_errors():
    with pytest.raises(ValueError, match="Expected at least `2` clusters, found `1`"):
        NhoodPlan(np.array([0, 1]), np.array([0]), 1)
    plan = NhoodPlan(np.array([0, 1, 2]), np.array([1, 0]), 2)
    with pytest.raises(ValueError, match="n_cls"):
        plan.count(np.array([0, 5]))
    with pytest.raises(sq.SquidpyB200Error, match="set_base"):
        plan.upload(spawn_states(0, 2))
    # the kernels index the label arrays with the CSR columns: out-of-range / negative columns and a non-monotone indptr are
    # rejected when the graph is created (checked on the device, together with the symmetry test)
    with pytest.raises(ValueError, match="invalid CSR"):
        NhoodPlan(np.array([0, 1, 2, 3]), np.array([1, 7, 0]), 2)
    with pytest.raises(ValueError, match="invalid CSR"):
        NhoodPlan(np.array([0, 1, 2, 3], dtype=np.int32), np.array([1, -1, 0], dtype=np.int32), 2)
    with pytest.raises(ValueError, match="invalid CSR"):
        NhoodPlan(np.array([0, 2, 1, 3]), np.array([1, 2, 0]), 2)
    long_row = np.concatenate([np.arange(1, 101), [500]]).astype(np.int64)  # > 64 entries: no symmetry test, still validated
    with pytest.raises(ValueError, match="invalid CSR"):
        NhoodPlan(np.concatenate([[0], np.full(200, 101)]), long_row, 2)
    with pytest.raises(ValueError, match="Negative CSR index"):
        NhoodPlan(np.array([0, 1, 2]), np.array([1, -1], dtype=np.int64), 2)


@pytest.mark.parametrize("algo,threads,q", [(1, 128, 4), (1, 256, 4), (1, 512, 4), (1, 1024, 4), (2, 512, 1), (2, 512, 2), (2, 512, 4),
                                             (7, 128, 4), (7, 256, 4), (7, 256, 8), (7, 512, 2), (7, 512, 4), (7, 512, 8), (7, 1024, 2), (7, 1024, 4)])
@pytest.mark.parametrize("n", [2, 3, 5, 33, 100, 1000, 1025, 5041, 70001])
def test_shuffle_is_numpy_exact(algo, threads, q, n):
    """Shuffled label vectors equal numpy Generator.shuffle of the same spawned generators (oracle = exact replay,
    pinned to numpy in tests/test_oracle_golden.py)."""
    g = sp.csr_matrix((np.ones(n - 1, np.float32), (np.arange(n - 1), np.arange(1, n))), shape=(n, n))
    n_cls = 251
    base = (np.arange(n) % n_cls).astype(np.uint32)
    plan = _plan(g, n_cls)
    plan.set_option("shuffle_algo", algo)
    plan.set_option("shuffle_threads", threads)
    plan.set_option("shuffle_r" if algo == 7 else "shuffle_q", q)
    plan.set_base(base)
    P = 7
    st = spawn_states(1234 + n, P)
    plan.upload(st)
    got = plan.shuffled_labels(0, P)
    np.testing.assert_array_equal(got, ref.shuffle_labels(base, st))


@pytest.mark.parametrize("algo,threads,r", [(1, 512, 4), (2, 512, 4), (7, 1024, 2), (7, 512, 8), (-1, 512, 4)])
def test_shuffle_uint16_labels(algo, threads, r):
    """More than 256 categories: 16-bit label arrays through every replay variant (incl. the shared-memory low part of the
    default, which then holds half as many elements), with library segments."""
    n = 90001
    g = sp.csr_matrix((np.ones(n - 1, np.float32), (np.arange(n - 1), np.arange(1, n))), shape=(n, n))
    n_cls = 300
    base = (np.arange(n) * 7 % n_cls).astype(np.uint32)
    lib = (np.arange(n) % 2).astype(np.int32)
    plan = _plan(g, n_cls)
    plan.set_option("shuffle_algo", algo)
    plan.set_option("shuffle_threads", threads)
    plan.set_option("shuffle_r" if algo == 7 else "shuffle_q", r)
    if algo == 7:
        plan.set_option("shuffle_low", -1)
    P = 300 if algo == -1 else 5  # auto picks the two-kernel list replay only for more than 2 x SM permutations
    st = spawn_states(11, P)
    plan.set_base(base)
    plan.upload(st)
    np.testing.assert_array_equal(plan.shuffled_labels(P - 3, P), ref.shuffle_labels(base, st[P - 3 :]))
    plan.set_base(base, lib, 2)
    plan.upload(st)
    np.testing.assert_array_equal(plan.shuffled_labels(0, 2), ref.shuffle_labels(base, st[:2], lib, 2))


@pytest.mark.parametrize("q", [2, 4, 8])
@pytest.mark.parametrize("n", [9, 257, 1000, 4099, 70001])
def test_target_generation_batch_sizes(q, n):
    """Swap-target generation of the two-kernel replay (128 / 256 raw values per batch).  Small arrays are the hard case for
    its acceptance fixed point: a window covers a quarter of the remaining range, so many candidates depend on their rank."""
    g = sp.csr_matrix((np.ones(n - 1, np.float32), (np.arange(n - 1), np.arange(1, n))), shape=(n, n))
    base = (np.arange(n) % 113).astype(np.uint32)
    st = spawn_states(900 + n, 24)
    exp = ref.shuffle_labels(base, st)
    plan = _plan(g, 113)
    plan.set_option("shuffle_algo", 7)
    plan.set_option("shuffle_q", q)
    plan.set_base(base)
    plan.upload(st)
    np.testing.assert_array_equal(plan.shuffled_labels(0, 24), exp)


@pytest.mark.parametrize("algo", [7])
@pytest.mark.parametrize("low", [0, 1024, 50000, -1])
def test_two_kernel_replay_low_part(low, algo):
    """algo 7 can keep the first `low` positions of every label array in shared memory: same permutations for any split."""
    n = 70001
    g = sp.csr_matrix((np.ones(n - 1, np.float32), (np.arange(n - 1), np.arange(1, n))), shape=(n, n))
    base = (np.arange(n) % 97).astype(np.uint32)
    lib = (np.arange(n) % 3).astype(np.int32)
    plan = _plan(g, 97)
    plan.set_option("shuffle_algo", algo)
    plan.set_option("shuffle_low", low)
    st = spawn_states(77, 5)
    plan.set_base(base)
    plan.upload(st)
    np.testing.assert_array_equal(plan.shuffled_labels(0, 5), ref.shuffle_labels(base, st))
    plan.set_base(base, lib, 3)
    plan.upload(st)
    np.testing.assert_array_equal(plan.shuffled_labels(0, 5), ref.shuffle_labels(base, st, lib, 3))


@pytest.mark.parametrize("algo", [1, 2, 7])
def test_shuffle_library_groups(algo):
    n = 4000
    g = synth.hex_graph(40, 100)
    rng = np.random.default_rng(3)
    base = rng.integers(0, 9, n).astype(np.uint32)
    lib = rng.integers(0, 4, n).astype(np.int32)
    lib[:7] = 3  # unbalanced, interleaved membership
    plan = _plan(g, 9)
    plan.set_option("shuffle_algo", algo)
    plan.set_base(base, lib, 5)  # category 4 is empty
    st = spawn_states(99, 6)
    plan.upload(st)
    np.testing.assert_array_equal(plan.shuffled_labels(0, 6), ref.shuffle_labels(base, st, lib, 5))
    np.testing.assert_array_equal(plan.permute(st), ref.nhood_perm_counts(g.indptr, g.indices, base, 9, st, lib, 5))


@pytest.mark.parametrize("n_cls,P", [(10, 100), (30, 70), (64, 33), (300, 5)])
def test_perm_counts_vs_oracle(n_cls, P):
    g = synth.hex_graph(71, 71)
    base = np.random.default_rng(0).integers(0, n_cls, g.shape[0]).astype(np.uint32)
    plan = _plan(g, n_cls)
    plan.set_base(base)
    st = spawn_states(42, P)
    got = plan.permute(st)
    assert got.dtype == np.uint32 and got.shape == (P, n_cls, n_cls)
    np.testing.assert_array_equal(got, ref.nhood_perm_counts(g.indptr, g.indices, base, n_cls, st))


def test_perm_chunking_and_resident_api():
    g = synth.knn_graph(np.random.default_rng(1).random((3000, 2)), 6)
    base = np.random.default_rng(2).integers(0, 5, 3000).astype(np.uint32)
    st = spawn_states(7, 70)
    plan = _plan(g, 5)
    plan.set_base(base)
    full = plan.permute(st)
    plan.set_option("perm_chunk", 32)  # 3 chunks
    np.testing.assert_array_equal(plan.permute(st), full)
    plan.upload(st)
    plan.run_async()
    plan.run_async()  # re-running is idempotent
    np.testing.assert_array_equal(plan.download(), full)
    np.testing.assert_array_equal(full, ref.nhood_perm_counts(g.indptr, g.indices, base, 5, st))
    assert plan.bytes_per_perm == 4 * g.nnz + 4 * 3001 + 8 * 3000 + 4 * 25


def test_api_matches_reference_golden(golden_dummy, dummy_adata):
    """Public API on the reference's dummy_adata recipe: z-scores IDENTICAL to the reference (same permutations, same
    float64 mean/std), counts bit-exact, keys/dtypes as in reference tests/graph/test_nhood.py:20-25."""
    res = sq.gr.nhood_enrichment(dummy_adata, "cluster", n_perms=20, seed=42, copy=True)
    np.testing.assert_array_equal(res.counts, golden_dummy["nhood_count"])
    np.testing.assert_array_equal(res.zscore, golden_dummy["nhood_z"])
    assert res.zscore[0, 0] == 0.4957188836779417  # SURVEY.md Appendix A, KAT-2
    out = sq.gr.nhood_enrichment(dummy_adata, "cluster", library_key="library", n_perms=20, seed=42)
    assert out is None
    d = dummy_adata.uns["cluster_nhood_enrichment"]
    assert d["zscore"].dtype == np.float64 and d["count"].dtype == np.uint32 and d["zscore"].shape == (3, 3)
    np.testing.assert_array_equal(d["zscore"], golden_dummy["nhood_lib_z"])
    np.testing.assert_array_equal(d["count"], golden_dummy["nhood_lib_count"])


def test_api_cfg1_visium_grid_golden(golden_cfg1):
    """BASELINE.json configs[0]: 5 041-spot Visium grid, 10 clusters, n_perms=100 — against the reference's output."""
    g = synth.hex_graph(71, 71)
    assert g.nnz == int(golden_cfg1["nnz"])
    lab = pd.Series(pd.Categorical.from_codes(golden_cfg1["codes"].astype(int), categories=[f"c{i:03d}" for i in range(10)]))
    ad = synth.make_adata(synth.hex_coords(71, 71), g, lab)
    res = sq.gr.nhood_enrichment(ad, "cluster", n_perms=100, seed=42, copy=True)
    np.testing.assert_array_equal(res.counts, golden_cfg1["nhood_count"])
    np.testing.assert_array_equal(res.zscore, golden_cfg1["nhood_z"])


def test_device_stats_are_numpy_bitwise():
    """Mean / std over the permutations computed on the device equal numpy's float64 mean/std of the downloaded counts BIT FOR
    BIT (same operation order, no FMA contraction): the z-scores of the single-GPU path are the reference's."""
    g = synth.hex_graph(61, 47)
    n_cls = 12
    lab = np.random.default_rng(2).integers(0, n_cls, g.shape[0]).astype(np.uint32)
    for P in (1, 2, 7, 333, 1000):
        plan = _plan(g, n_cls)
        plan.set_base(lab)
        plan.upload(spawn_states(5, P))
        plan.run_async()
        mean, std = plan.stats()
        perms = plan.download().astype(np.float64)
        assert mean.tobytes() == perms.mean(axis=0).tobytes()
        assert std.tobytes() == perms.std(axis=0).tobytes()
    with pytest.raises(sq.SquidpyB200Error, match="nothing has run"):
        _plan(g, n_cls).stats()


def test_device_chained_stats_are_numpy_bitwise():
    """The multi-GPU form of the statistics (exact integer sums + variance accumulation continued from a running value):
    two plans holding consecutive shards of the permutations reproduce numpy's mean/std of all of them bit for bit."""
    g = synth.hex_graph(41, 37)
    n_cls = 9
    lab = np.random.default_rng(4).integers(0, n_cls, g.shape[0]).astype(np.uint32)
    P, cut = 301, 120
    st = spawn_states(8, P)
    plans, counts = [], []
    for lo, hi in ((0, cut), (cut, P)):
        plan = _plan(g, n_cls)
        plan.set_base(lab)
        plan.upload(st[lo:hi])
        plan.run_async()
        plans.append(plan)
        counts.append(plan.download())
    full = np.concatenate(counts).astype(np.float64)
    total = plans[0].sums() + plans[1].sums()
    np.testing.assert_array_equal(total, np.concatenate(counts).sum(axis=0, dtype=np.int64))
    mean = total.astype(np.float64) / P
    assert mean.tobytes() == full.mean(axis=0).tobytes()
    acc = plans[1].var_chain(mean, plans[0].var_chain(mean, np.zeros_like(mean)))
    assert np.sqrt(acc / P).tobytes() == full.std(axis=0).tobytes()


def test_api_reproducibility(dummy_adata):
    # reference tests/graph/test_nhood.py:41-59
    a = sq.gr.nhood_enrichment(dummy_adata, "cluster", n_perms=30, seed=42, copy=True)
    b = sq.gr.nhood_enrichment(dummy_adata, "cluster", n_perms=30, seed=42, copy=True, n_jobs=2, backend="threading")
    c = sq.gr.nhood_enrichment(dummy_adata, "cluster", n_perms=30, seed=43, copy=True)
    np.testing.assert_array_equal(a.zscore, b.zscore)
    np.testing.assert_array_equal(a.counts, c.counts)
    assert not np.allclose(a.zscore, c.zscore)


def test_full_size_1m_spots():
    """BASELINE.json configs[1] shape (1M spots, 30 clusters, k=6): direct parity on a few permutations plus
    size-independent properties on all of them."""
    g = synth.hex_graph(1000, 1000)
    n = g.shape[0]
    base = np.random.default_rng(0).integers(0, 30, n).astype(np.uint32)
    plan = _plan(g, 30)
    np.testing.assert_array_equal(plan.count(base), ref.nhood_count(g.indptr, g.indices, base, 30))
    plan.set_base(base)
    P = 48
    st = spawn_states(0, P)
    got = plan.permute(st)
    np.testing.assert_array_equal(got[:6], ref.nhood_perm_counts(g.indptr, g.indices, base, 30, st[:6]))
    assert (got.reshape(P, -1).sum(axis=1, dtype=np.int64) == g.nnz).all()  # every stored entry counted once
    np.testing.assert_array_equal(got, got.transpose(0, 2, 1))  # symmetric graph -> symmetric counts
    # every replay at full size, incl. several permutations per CTA
    for algo in (1, 2, 7):
        plan.set_option("shuffle_algo", algo)
        plan.set_option("shuffle_ctas", 16)
        np.testing.assert_array_equal(plan.permute(st), got)
    plan.set_option("shuffle_algo", -1)
    plan.set_option("shuffle_ctas", 0)
    lab = plan.shuffled_labels(40, 42)
    np.testing.assert_array_equal(np.sort(lab, axis=1), np.sort(np.broadcast_to(base, lab.shape), axis=1))  # a permutation
    np.testing.assert_array_equal(lab, ref.shuffle_labels(base, st[40:42]))


def test_buffered_generator_states_are_rejected():
    """A generator that already handed out half of a 64-bit draw (has_uint32 = 1) cannot be replayed from (state, inc) alone:
    the C ABI refuses it instead of producing different permutations."""
    g = synth.hex_graph(9, 9)
    plan = NhoodPlan(g.indptr, g.indices, 3)
    plan.set_base(np.random.default_rng(0).integers(0, 3, g.shape[0]).astype(np.uint32))
    st = spawn_states(1, 4)
    st[2, 4] = 1
    with pytest.raises(NotImplementedError, match="has_uint32"):
        plan.upload(st)
    plan.upload(spawn_states(1, 4))  # the handle stays usable
    assert plan.permute(spawn_states(1, 4)).shape == (4, 3, 3)
    plan.close()


def test_set_option_rejects_unknown_replays():
    """shuffle_algo takes -1 (auto), 1, 2 and 7; anything else is refused when it is set, and the plan keeps working."""
    g = synth.hex_graph(12, 12)
    base = np.random.default_rng(0).integers(0, 4, g.shape[0]).astype(np.uint32)
    plan = _plan(g, 4)
    plan.set_base(base)
    for algo in (-2, 0, 3, 4, 5, 6, 8, 9):
        with pytest.raises(ValueError, match="shuffle_algo must be"):
            plan.set_option("shuffle_algo", algo)
    with pytest.raises(ValueError, match="unknown key 'shuffle_region'"):
        plan.set_option("shuffle_region", 0)
    plan.set_option("shuffle_algo", -1)
    st = spawn_states(1, 3)
    np.testing.assert_array_equal(plan.permute(st), ref.nhood_perm_counts(g.indptr, g.indices, base, 4, st))
