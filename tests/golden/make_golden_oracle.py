"""Generates tests/golden/oracle_reference.npz: what the UNMODIFIED reference code returns for the seeded inputs of
tests/test_oracle_vs_reference.py (nhood count function + permutation helper, ``_occur_count`` / ``_co_occurrence_helper``,
the ``_interaction_matrix`` numba kernel), run through the stub-import loader ``oracle/_refload.py``.  Only runnable where the
reference sources are present; the output is committed.  The GridBuilder graph that test checks is ``grid6_hex`` of
tests/golden/graphs.npz.

    python tests/golden/make_golden_oracle.py
"""

from __future__ import annotations

import os
import sys

import numpy as np
import pandas as pd
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tools import synth  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle_reference.npz")
NHOOD_CASES = [(2, False), (7, False), (30, True)]
NHOOD_PERMS, NHOOD_SEED = 12, 11


def nhood_case(n_cls, libs):
    """(indptr, indices, labels, libraries or None) of the nhood case; shared with tests/test_oracle_vs_reference.py"""
    g = synth.hex_graph(37, 41)
    n = g.shape[0]
    lab = np.random.default_rng(n_cls).integers(0, n_cls, n).astype(np.uint32)
    libraries = pd.Series(pd.Categorical(np.random.default_rng(1).integers(0, 3, n).astype(str))) if libs else None
    return g.indptr.astype(np.uint32), g.indices.astype(np.uint32), lab, libraries


def cooc_case():
    rr = np.random.default_rng(5)
    pts = (rr.random((1500, 2)) * 300).astype(np.float32)
    lb = rr.integers(0, 5, 1500).astype(np.int32)
    iv = np.linspace(1, 200, 20, dtype=np.float32)
    return pts, lb, iv


def interaction_cases():
    """(name, graph, codes, k) of the random-graph interaction-matrix cases"""
    rng = np.random.default_rng(0)
    out = []
    for n, dens, k in ((200, 0.05, 5), (1500, 0.004, 12)):
        a = sp.random(n, n, density=dens, format="csr", random_state=int(rng.integers(1 << 30)), dtype=np.float32)
        out.append((f"n{n}", a, rng.integers(0, k, n), k))
    return out


def main():
    from oracle import _refload

    m = _refload.load()
    nh, pp = m["nh"], m["pp"]
    out = {"meta": np.array(f"numpy {np.__version__}; reference squidpy (be17fcf6) gr/_nhood.py, gr/_ppatterns.py")}
    for n_cls, libs in NHOOD_CASES:
        ptr, ind, lab, libraries = nhood_case(n_cls, libs)
        fn = nh._create_function(n_cls)
        gens = m["utils"].spawn_generators(NHOOD_SEED, NHOOD_PERMS)
        out[f"nhood{n_cls}_count"] = fn(ind, ptr, lab)
        out[f"nhood{n_cls}_perms"] = nh._nhood_enrichment_helper(list(range(NHOOD_PERMS)), fn, ind, ptr, lab, libraries, n_cls, gens).astype(np.uint32)
    pts, lb, iv = cooc_case()
    out["cooc_counts"] = pp._occur_count(pts[:, 0].copy(), pts[:, 1].copy(), iv[1:] ** 2, lb, 1500, 5, 19)
    out["cooc_occ"] = pp._co_occurrence_helper(pts[:, 0].copy(), pts[:, 1].copy(), iv, lb)
    for name, a, codes, k in interaction_cases():
        for weights in (False, True):
            data = a.data if weights else np.broadcast_to(1, shape=len(a.data))
            exp = np.zeros((k, k), dtype=float)
            nh._interaction_matrix(np.ascontiguousarray(data), a.indices, a.indptr, codes, exp)
            out[f"interaction_{name}_w{int(weights)}"] = exp
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, os.path.getsize(OUT))


if __name__ == "__main__":
    main()
