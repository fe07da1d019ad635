"""Generates tests/golden/graphs.npz: outputs of the UNMODIFIED reference graph builders
(the reference's ``src/squidpy/gr/neighbors.py``: KNNBuilder, RadiusBuilder, GridBuilder incl. post-processing and the
``library_key`` block-diagonal combination) on seeded inputs, through the stub-import loader ``oracle/_refload.py``.
Only runnable where the reference sources are present; the output is committed.  Read it with :func:`load`: float64
distances are stored as the bitwise XOR with ``sqrt(dx*dx + dy*dy)`` of the coordinates (zero where they agree, which
compresses to almost nothing), and :func:`load` restores the reference's values bit for bit.

    python tests/golden/make_golden_graphs.py
"""

from __future__ import annotations

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import _refload  # noqa: E402
from tools import synth  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
PATH = os.path.join(OUT, "graphs.npz")


def cases():
    """name -> (coords, builder class name, kwargs); shared with tests/test_gpu_graphs.py"""
    rng = np.random.default_rng(7)
    uni = rng.random((3000, 2)) * 1000.0
    clustered = (rng.random((12, 2)) * 800.0)[rng.integers(0, 12, 2500)] + rng.normal(0.0, 30.0, (2500, 2))  # clusters, no exact ties
    hexg = synth.hex_coords(23, 31)
    sq = np.stack(np.meshgrid(np.arange(12, dtype=float), np.arange(9, dtype=float)), -1).reshape(-1, 2) * 10.0
    c = {
        "knn6_uniform": (uni, "KNNBuilder", dict(n_neighs=6)),
        "knn15_clustered": (clustered, "KNNBuilder", dict(n_neighs=15)),
        "knn4_diag_pct_spectral": (uni[:800], "KNNBuilder", dict(n_neighs=4, set_diag=True, percentile=90.0, transform="spectral")),
        "knn6_cosine": (uni[:500], "KNNBuilder", dict(n_neighs=6, transform="cosine")),
        "grid6_hex": (hexg, "GridBuilder", dict(n_neighs=6)),
        "grid6_hex_rings2_diag": (hexg, "GridBuilder", dict(n_neighs=6, n_rings=2, set_diag=True)),
        "grid4_square": (sq, "GridBuilder", dict(n_neighs=4)),
        "grid6_uniform": (uni[:1500], "GridBuilder", dict(n_neighs=6)),
        "radius_uniform": (uni, "RadiusBuilder", dict(radius=25.0)),
        "radius_interval_spectral": (clustered, "RadiusBuilder", dict(radius=(5.0, 20.0), transform="spectral")),
    }
    return c


def _predicted_bits(co, indptr, indices):
    """bits of the float64 sqrt(dx*dx + dy*dy) of every stored entry (row of indptr, column in indices)"""
    r = np.repeat(np.arange(len(indptr) - 1), np.diff(indptr))
    d = co[r] - co[indices]
    return np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]).view(np.uint64)


def _coords(gold, prefix):
    return gold["lib_coords"] if prefix == "lib" else cases()[prefix][0]


def _pack(out):
    """float64 `<prefix>_dst_data` -> `<prefix>_dst_xor`: the bits XOR the predicted distance"""
    for k in [k for k in out if k.endswith("_dst_data") and out[k].dtype == np.float64]:
        p = k[: -len("_dst_data")]
        out[f"{p}_dst_xor"] = out.pop(k).view(np.uint64) ^ _predicted_bits(_coords(out, p), out[f"{p}_dst_indptr"], out[f"{p}_dst_indices"])
    return out


def load() -> dict:
    """graphs.npz with every `<prefix>_dst_data` as the reference returned it"""
    gold = dict(np.load(PATH, allow_pickle=False))
    for k in [k for k in gold if k.endswith("_dst_xor")]:
        p = k[: -len("_dst_xor")]
        gold[f"{p}_dst_data"] = (gold.pop(k) ^ _predicted_bits(_coords(gold, p), gold[f"{p}_dst_indptr"], gold[f"{p}_dst_indices"])).view(np.float64)
    return gold


def main():
    import scipy
    import sklearn

    nb = _refload.load()["nb"]
    # numba cannot type scipy's csr_matrix here (the reference relies on an extension that is not installed): run the
    # reference's own helper un-jitted (same code, interpreted)
    nb._csr_bilateral_diag_scale_helper = nb._csr_bilateral_diag_scale_helper.py_func
    out = {"meta": np.array(f"numpy {np.__version__}; scipy {scipy.__version__}; sklearn {sklearn.__version__}; reference squidpy (be17fcf6) gr/neighbors.py")}
    for name, (co, cls, kw) in cases().items():
        adj, dst = getattr(nb, cls)(**kw).build(co.copy())
        for tag, m in (("adj", adj), ("dst", dst)):
            m = m.tocsr()
            m.sort_indices()
            out[f"{name}_{tag}_indptr"], out[f"{name}_{tag}_indices"], out[f"{name}_{tag}_data"] = m.indptr, m.indices, m.data
    # library_key: two interleaved libraries -> block diagonal in the original order (GraphBuilderCSR.combine)
    rng = np.random.default_rng(11)
    co = rng.random((400, 2)) * 300.0
    codes = rng.integers(0, 2, 400)
    b = nb.KNNBuilder(n_neighs=5)
    mats, ixs = [], []
    for c in range(2):
        idx = np.where(codes == c)[0]
        mats.append(b.build(np.ascontiguousarray(co[idx])))
        ixs.extend(idx.tolist())
    adj, dst = b.combine(mats, ixs)
    out["lib_coords"], out["lib_codes"] = co, codes
    for tag, m in (("adj", adj), ("dst", dst)):
        m = m.tocsr()
        m.sort_indices()
        out[f"lib_{tag}_indptr"], out[f"lib_{tag}_indices"], out[f"lib_{tag}_data"] = m.indptr, m.indices, m.data
    np.savez_compressed(PATH, **_pack(out))
    print("wrote graphs.npz", {k: v.shape for k, v in out.items() if k.endswith("adj_data")})


if __name__ == "__main__":
    main()
