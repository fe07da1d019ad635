"""CPU oracle for the squidpy spatial-statistics hot path — TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl reference`` legs of
``bench.py`` may import this package.  The product package ``squidpy_b200`` never does (a test enforces it).

Contents
--------
* ``c/oracle.c`` + ``liboracle.so`` — C restatement of the reference algorithms (nhood count + exact numpy
  PCG64 ``Generator.shuffle`` replay, co-occurrence counts, Ripley pair counts, Moran's I / Geary's C); every
  function cites the reference ``file:line`` it follows.
* ``ref.py`` — numpy-level wrappers around the C library plus the float/host post-processing of each
  reference function (z-scores, occ ratio, L estimate, analytic p-values) restated in numpy.
* ``_refload.py`` — stub-import loader that runs the UNMODIFIED reference modules from a checkout of the reference
  sources (``$SQUIDPY_REF``); used only to generate ``tests/golden/*.npz`` (``tests/golden/make_golden*.py``), against
  which ``tests/test_oracle_vs_reference.py`` and ``tests/test_oracle_golden.py`` pin the restatement.

Pinning status: nhood_enrichment, co_occurrence, Ripley L/F/G and the analytic moments are pinned against the
running reference code and against golden vectors generated from it (SURVEY.md Appendix A).  Moran's I / Geary's C
values are **parity unpinned**: the arithmetic lives in scanpy (absent here, un-pinned dependency) and no
reference test holds a numeric value for it; the restatement follows scanpy's published algorithm and is
cross-checked against an independent scipy.sparse formulation only.
"""

from __future__ import annotations

import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "liboracle.so")
_lib = None


def build(force: bool = False) -> str:
    """Compile ``c/oracle.c`` -> ``liboracle.so`` with the committed Makefile."""
    src = os.path.join(_HERE, "c", "oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.run(["make", "-C", _HERE, "-B", "liboracle.so"], check=True, capture_output=True)
    return _LIB_PATH


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        _lib = ctypes.CDLL(_LIB_PATH)
    return _lib
