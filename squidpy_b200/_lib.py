"""ctypes binding of ``libsquidpy_b200.so`` (C ABI declared in ``include/squidpy_b200.h``).

The CUDA library is the product: there is NO CPU fallback.  If the shared library is missing, was built for
another ABI version, or no CUDA device is present, every entry point fails loudly.
"""

from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsquidpy_b200.so")
ABI_VERSION = 3

_lock = threading.Lock()
_lib: C.CDLL | None = None

c_void_pp = C.POINTER(C.c_void_p)


class SquidpyB200Error(RuntimeError):
    """Raised when the CUDA library reports a failure."""


def _ptr(arr: np.ndarray | None):
    return None if arr is None else arr.ctypes.data_as(C.c_void_p)


# name -> (restype, argtypes); every symbol of include/squidpy_b200.h
_SIGNATURES: dict[str, tuple] = {
    "sqb_abi_version": (C.c_int, []),
    "sqb_last_error": (C.c_char_p, []),
    "sqb_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "sqb_ctx_create": (C.c_int, [C.c_int, C.c_void_p, c_void_pp]),
    "sqb_ctx_destroy": (C.c_int, [C.c_void_p]),
    "sqb_ctx_sync": (C.c_int, [C.c_void_p]),
    "sqb_ctx_stream": (C.c_int, [C.c_void_p, c_void_pp]),
    "sqb_ctx_sm_count": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "sqb_ctx_launch_count": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "sqb_ctx_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "sqb_ctx_profile_reset": (C.c_int, [C.c_void_p]),
    "sqb_ctx_profile_get": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "sqb_host_alloc": (C.c_int, [C.c_size_t, c_void_pp]),
    "sqb_host_free": (C.c_int, [C.c_void_p]),
    "sqb_nhood_create": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int, c_void_pp]),
    "sqb_nhood_destroy": (C.c_int, [C.c_void_p]),
    "sqb_nhood_count": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "sqb_nhood_set_base": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "sqb_nhood_permute": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "sqb_nhood_permute_upload": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "sqb_nhood_permute_upload_philox": (C.c_int, [C.c_void_p, C.c_uint64, C.c_int64, C.c_int64]),
    "sqb_nhood_permute_run_async": (C.c_int, [C.c_void_p]),
    "sqb_nhood_permute_download": (C.c_int, [C.c_void_p, C.c_void_p]),
    "sqb_nhood_permute_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "sqb_interaction_matrix": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                          C.c_int, C.c_void_p, C.c_void_p]),
    "sqb_nhood_permute_sums": (C.c_int, [C.c_void_p, C.c_void_p]),
    "sqb_nhood_permute_var_chain": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sqb_nhood_permute_stats_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "sqb_nhood_permute_sums_dev": (C.c_int, [C.c_void_p, C.c_void_p]),
    "sqb_nhood_permute_var_chain_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sqb_nhood_permute_counts_dev": (C.c_int, [C.c_void_p, C.c_void_p]),
    "sqb_nhood_stats_rows_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]),
    "sqb_nhood_shuffled_labels": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]),
    "sqb_nhood_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    "sqb_nhood_bytes_per_perm": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "sqb_autocorr_create": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, c_void_pp]),
    "sqb_autocorr_destroy": (C.c_int, [C.c_void_p]),
    "sqb_autocorr_load_dense": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64]),
    "sqb_autocorr_load_csr": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64]),
    "sqb_autocorr_load_csr_cols": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int64]),
    "sqb_autocorr_run_async": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "sqb_autocorr_download": (C.c_int, [C.c_void_p, C.c_void_p]),
    "sqb_autocorr_run_perms": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p]),
    "sqb_autocorr_dense": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_void_p]),
    "sqb_autocorr_csr": (
        C.c_int,
        [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_void_p],
    ),
    "sqb_ligrec_counts": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                    C.c_void_p, C.c_void_p]),
    "sqb_sepal": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64,
                            C.c_int, C.c_double, C.c_double, C.c_void_p]),
    "sqb_knn_2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sqb_radius_2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]),
    "sqb_cooc_counts": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p],
    ),
    "sqb_pair_counts_f64": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p],
    ),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def load() -> C.CDLL:
    """Load the CUDA library (once).  Raises :class:`SquidpyB200Error` if it is missing — never falls back."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise SquidpyB200Error(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C squidpy_b200/csrc`).  squidpy_b200 has no CPU fallback."
            )
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            try:
                fn = getattr(lib, name)
            except AttributeError as e:  # pragma: no cover
                raise SquidpyB200Error(f"{LIB_PATH} does not export `{name}` (stale build?)") from e
            fn.restype = res
            fn.argtypes = args
        v = lib.sqb_abi_version()
        if v != ABI_VERSION:
            raise SquidpyB200Error(f"{LIB_PATH} has ABI version {v}, expected {ABI_VERSION}: rebuild")
        _lib = lib
        return lib


def check(rc: int, exc: type[Exception] | None = None) -> None:
    """Translate a negative status into a Python exception (ValueError for invalid arguments)."""
    if rc == 0:
        return
    msg = load().sqb_last_error().decode("utf-8", "replace")
    if exc is not None:
        raise exc(msg)
    if rc == -1:
        raise ValueError(msg)
    if rc == -3:
        raise MemoryError(msg)
    if rc == -4:
        raise NotImplementedError(msg)
    raise SquidpyB200Error(f"[status {rc}] {msg}")


def device_count() -> int:
    n = C.c_int(0)
    check(load().sqb_device_count(C.byref(n)))
    return n.value


KCLASS = {
    "fill": 0,
    "shuffle": 1,
    "transpose": 2,
    "count": 3,
    "autocorr_prep": 4,
    "autocorr_main": 5,
    "autocorr_final": 6,
    "pairs": 7,
    "misc": 8,
}


class Context:
    """One CUDA device + one stream.  ``stream`` may be a raw ``cudaStream_t`` value (e.g.
    ``torch.cuda.current_stream().cuda_stream``) so that the caller's CUDA events see the library's kernels."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self._lib = load()
        h = C.c_void_p()
        check(self._lib.sqb_ctx_create(int(device), C.c_void_p(stream) if stream else None, C.byref(h)))
        self._h = h
        self.device = int(device)
        self.lock = threading.RLock()  # held by the sq.gr.* calls while they use this context's stream / scratch buffers

    @property
    def handle(self) -> C.c_void_p:
        if self._h is None:
            raise SquidpyB200Error("context already destroyed")
        return self._h

    def sync(self) -> None:
        check(self._lib.sqb_ctx_sync(self.handle))

    @property
    def stream(self) -> int:
        s = C.c_void_p()
        check(self._lib.sqb_ctx_stream(self.handle, C.byref(s)))
        return s.value or 0

    @property
    def sm_count(self) -> int:
        n = C.c_int()
        check(self._lib.sqb_ctx_sm_count(self.handle, C.byref(n)))
        return n.value

    @property
    def launches(self) -> int:
        n = C.c_int64()
        check(self._lib.sqb_ctx_launch_count(self.handle, C.byref(n)))
        return n.value

    def profile(self, enable: bool) -> None:
        check(self._lib.sqb_ctx_profile(self.handle, int(enable)))

    def profile_reset(self) -> None:
        check(self._lib.sqb_ctx_profile_reset(self.handle))

    def profile_get(self, kclass: str | int) -> tuple[float, int]:
        k = KCLASS[kclass] if isinstance(kclass, str) else int(kclass)
        ms, n = C.c_double(), C.c_int64()
        check(self._lib.sqb_ctx_profile_get(self.handle, k, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def close(self) -> None:
        if self._h is not None:
            self._lib.sqb_ctx_destroy(self._h)
            self._h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass


_default_ctx: dict[int, Context] = {}
_default_ctx_lock = threading.Lock()


def default_context(device: int | None = None) -> Context:
    """Per-device shared context.  ``device=None`` resolves to ``$LOCAL_RANK`` (one process per GPU) or 0.
    The context (stream, scratch buffers, staging ring) is shared by every ``sq.gr.*`` call on that device: the calls hold
    ``ctx.lock`` while they use it, so concurrent calls from several Python threads serialise instead of interleaving."""
    if device is None:
        device = int(os.environ.get("SQB_DEVICE", os.environ.get("LOCAL_RANK", "0")))
        n = device_count()
        device = device % max(n, 1)
    with _default_ctx_lock:
        if device not in _default_ctx:
            _default_ctx[device] = Context(device)
        return _default_ctx[device]


def set_default_context(ctx: Context | None, device: int | None = None) -> None:
    """Make ``ctx`` the context ``sq.gr.*`` uses on its device (e.g. one created on torch's current stream, so that CUDA
    events and NCCL collectives issued by the caller are ordered with the library's kernels); ``None`` removes it."""
    with _default_ctx_lock:
        if ctx is None:
            _default_ctx.pop(int(device or 0), None)
        else:
            _default_ctx[ctx.device] = ctx


def pinned_empty(shape, dtype) -> np.ndarray:
    """numpy array backed by page-locked host memory (freed when the array is garbage collected)."""
    lib = load()
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    p = C.c_void_p()
    check(lib.sqb_host_alloc(max(n, 1), C.byref(p)))
    buf = (C.c_char * max(n, 1)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    class _Owner:
        def __init__(self, ptr):
            self.ptr = ptr

        def __del__(self):
            try:
                lib.sqb_host_free(C.c_void_p(self.ptr))
            except Exception:
                pass

    _owners[id(buf)] = _Owner(p.value)
    import weakref

    weakref.finalize(buf, _owners.pop, id(buf), None)
    return arr


_owners: dict[int, object] = {}
