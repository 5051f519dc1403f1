"""ctypes binding of liblpvs.so -- the same C ABI the Julia shim ``ccall``s (include/lpvs.h).

There is no CPU fallback: if the shared library is missing, or no B200 is visible, the estimators raise.
"""
from __future__ import annotations

import ctypes as C
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LPVS_LIB") or os.path.join(_HERE, "liblpvs.so")  # LPVS_LIB: kernel-variant experiments only
HEADER_PATH = os.path.join(_HERE, "..", "include", "lpvs.h")

OK = 0
E_BAD_ARG, E_NOT_SPD, E_NONFINITE, E_CUDA, E_NCCL, E_UNSUPPORTED, E_NOMEM = -1, -2, -3, -4, -5, -6, -7
WIN_PSD, WIN_CSD, WIN_COHERE = 0, 1, 2
PROX_L1, PROX_L0, PROX_BALL_L0, PROX_GROUP_L2 = 0, 1, 2, 3
PHASE_AUTO, PHASE_CHAIN, PHASE_DIRECT, PHASE_CHAIN_REF, PHASE_STRUCTURED, PHASE_STRUCTURED_REF = 0, 1, 2, 3, 4, 5
OPT_PHASE_MODE, OPT_WINDOW_BATCH, OPT_JITTER, OPT_ADMM_CHECK_EVERY, OPT_ADMM_SYMV, OPT_TRSV_FLOW, OPT_SHARD_EXCHANGE, OPT_ADMM_M32 = 0, 1, 2, 3, 4, 5, 6, 7
INFO_JITTER = 1
INFO_QR = 2
INFO_DUAL = 3

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_i64p = C.POINTER(C.c_int64)
_vp = C.c_void_p

_PROTOS = {
    "lpvs_version": (C.c_int, []),
    "lpvs_device_count": (C.c_int, []),
    "lpvs_init": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "lpvs_destroy": (None, [_vp]),
    "lpvs_last_error": (C.c_char_p, [_vp]),
    "lpvs_set_option": (C.c_int, [_vp, C.c_int, C.c_double]),
    "lpvs_set_stream": (C.c_int, [_vp, _vp]),
    "lpvs_launch_count": (C.c_int64, [_vp]),
    "lpvs_last_gram_timing": (C.c_int, [_vp, _dp, _i64p, _dp]),
    "lpvs_last_call_ms": (C.c_int, [_vp, _dp]),
    "lpvs_dev_alloc": (C.c_int, [_vp, C.c_int64, C.POINTER(_vp)]),
    "lpvs_dev_free": (C.c_int, [_vp, _vp]),
    "lpvs_dev_upload": (C.c_int, [_vp, _vp, _vp, C.c_int64]),
    "lpvs_dev_download": (C.c_int, [_vp, _vp, _vp, C.c_int64]),
    "lpvs_sync": (C.c_int, [_vp]),
    "lpvs_release_workspace": (C.c_int, [_vp]),
    "lpvs_window_count": (C.c_int64, [C.c_int64, C.c_int, C.c_int]),
    "lpvs_gram_fourier": (C.c_int, [_vp, _vp, _vp, C.c_int64, _vp, C.c_int, _vp, _vp, _vp]),
    "lpvs_ls_spectral": (C.c_int, [_vp, _vp, _vp, C.c_int64, _vp, C.c_int, _vp, C.c_double, _vp, _ip]),
    "lpvs_ls_spectral_multi": (C.c_int, [_vp, _vp, C.c_int, C.c_int64, _vp, C.c_int64, _vp, C.c_int, _vp, C.c_double,
                                         _vp, _ip]),
    "lpvs_ls_spectral_multi_dev": (C.c_int, [_vp, _vp, C.c_int, C.c_int64, _vp, C.c_int64, _vp, C.c_int, _vp, C.c_double,
                                             _vp, _ip]),
    "lpvs_merge_windows": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, C.c_int, C.c_int64, _vp]),
    "lpvs_tls_spectral": (C.c_int, [_vp, _vp, _vp, C.c_int64, _vp, C.c_int, _vp, _ip]),
    "lpvs_ls_window_sums": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, C.c_int64, _vp, C.c_int, _vp, C.c_int, C.c_int,
                                      C.c_double, C.c_int64, C.c_int64, _vp, _ip]),
    "lpvs_ls_window_sums_dev": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, C.c_int64, _vp, C.c_int, _vp, C.c_int,
                                          C.c_int, C.c_double, C.c_int64, C.c_int64, _vp, _ip]),
    "lpvs_ls_window_sparse_sums": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, C.c_int64, _vp, C.c_int, _vp, C.c_int,
                                             C.c_int, C.c_int, C.c_double, C.c_double, C.c_int64, C.c_double,
                                             C.c_int64, C.c_int64, _vp, _vp, _vp, _ip]),
    "lpvs_ls_window_finalize": (C.c_int, [C.c_int, _vp, C.c_int, C.c_int64, _vp]),
    "lpvs_ls_window_matrix_sums": (C.c_int, [_vp, _vp, C.c_int, C.c_int64, _vp, C.c_int64, _vp, C.c_int, _vp, C.c_int,
                                             C.c_int, C.c_double, C.c_int64, C.c_int64, _vp, _ip]),
    "lpvs_ls_window_matrix_sums_dev": (C.c_int, [_vp, _vp, C.c_int, C.c_int64, _vp, C.c_int64, _vp, C.c_int, _vp,
                                                 C.c_int, C.c_int, C.c_double, C.c_int64, C.c_int64, _vp, _ip]),
    "lpvs_ls_window_matrix_finalize": (C.c_int, [C.c_int, _vp, C.c_int, C.c_int, C.c_int64, _vp]),
    "lpvs_ls_window_matrix_sparse_sums": (C.c_int, [_vp, _vp, C.c_int, C.c_int64, _vp, C.c_int64, _vp, C.c_int, _vp,
                                                    C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int64,
                                                    C.c_double, C.c_int64, C.c_int64, _vp, _vp, _vp, _ip]),
    "lpvs_ls_window_matrix_sparse_sums_dev": (C.c_int, [_vp, _vp, C.c_int, C.c_int64, _vp, C.c_int64, _vp, C.c_int,
                                                        _vp, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double,
                                                        C.c_int64, C.c_double, C.c_int64, C.c_int64, _vp, _vp, _vp,
                                                        _ip]),
    "lpvs_ls_window": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, C.c_int64, _vp, C.c_int, _vp, C.c_int, C.c_int,
                                 C.c_double, _vp, _i64p, _ip]),
    "lpvs_ls_spectral_lpv": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int64, _vp, C.c_int, C.c_int, C.c_double, C.c_int,
                                       C.c_int, _vp, _vp, _dp, _ip]),
    "lpvs_ls_windowpsd_lpv": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int64, _vp, C.c_int, C.c_int, C.c_int, C.c_int,
                                        C.c_double, C.c_int, C.c_int, _vp, _vp, _i64p, _ip]),
    "lpvs_ls_spectral_lpv_multi": (C.c_int, [_vp, _vp, C.c_int, C.c_int64, _vp, _vp, C.c_int64, _vp, C.c_int, C.c_int,
                                             C.c_double, C.c_int, C.c_int, _vp, _vp, _vp, _vp, _ip]),
    "lpvs_ls_windowpsd_lpv_multi": (C.c_int, [_vp, _vp, C.c_int, C.c_int64, _vp, _vp, C.c_int64, _vp, C.c_int, C.c_int,
                                              C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, _vp, _vp, _i64p, _ip]),
    "lpvs_admm_create_fourier": (C.c_int, [_vp, _vp, _vp, C.c_int64, _vp, C.c_int, _vp, C.c_int, C.c_double,
                                           C.c_double, _vp, C.c_int, C.c_double, C.POINTER(_vp)]),
    "lpvs_admm_create_lpv": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int64, _vp, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_double, C.c_double, C.POINTER(_vp)]),
    "lpvs_admm_run": (C.c_int, [_vp, C.c_int64, C.c_double, _i64p, _dp, _ip]),
    "lpvs_admm_shard_begin": (C.c_int, [_vp, C.c_int, C.c_int]),
    "lpvs_admm_shard_handle": (C.c_int, [_vp, _vp]),
    "lpvs_admm_shard_connect": (C.c_int, [_vp, _vp]),
    "lpvs_admm_size": (C.c_int, [_vp]),
    "lpvs_admm_get": (C.c_int, [_vp, _vp, _vp]),
    "lpvs_admm_result": (C.c_int, [_vp, _vp]),
    "lpvs_admm_last_timing": (C.c_int, [_vp, _dp, _dp]),
    "lpvs_admm_free": (None, [_vp]),
    "lpvs_ls_sparse_spectral": (C.c_int, [_vp, _vp, _vp, C.c_int64, _vp, C.c_int, _vp, C.c_int, C.c_double,
                                          C.c_double, C.c_int, C.c_double, C.c_int64, C.c_double, _vp, _i64p, _dp]),
    "lpvs_ls_sparse_spectral_lpv": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int64, _vp, C.c_int, C.c_int, C.c_int,
                                              C.c_int, C.c_double, C.c_double, C.c_int64, C.c_double, _vp, _i64p,
                                              _dp]),
    "lpvs_prox_fourier": (C.c_int, [_vp, C.c_int, C.c_double, C.c_double, _vp, C.c_int, C.c_int, _vp]),
    "lpvs_packed_size": (C.c_int64, [C.c_int]),
    "lpvs_gram_partial_dev": (C.c_int, [_vp, _vp, _vp, _vp, _vp, C.c_int64, _vp, C.c_int, _vp]),
    "lpvs_solve_packed_dev": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, C.c_double, _vp, _ip]),
}

_lib = None


def declared_symbols():
    """Every function include/lpvs.h declares (parsed from the header)."""
    with open(HEADER_PATH) as fh:
        src = fh.read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(lpvs_[a-z0-9_]+)\s*\(", src)))


def load():
    """dlopen liblpvs.so (no compute); raises if the extension was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _PROTOS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class LpvsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"liblpvs error {code}: {msg}")
        self.code = code


class NotPositiveDefinite(LpvsError):
    """Cholesky breakdown (Julia: PosDefException)."""


def raise_for(code, ctx_handle=None):
    if code == OK:
        return
    lib = load()
    msg = lib.lpvs_last_error(ctx_handle).decode() if ctx_handle else "no context"
    if code == E_BAD_ARG:
        raise ValueError(msg)  # Julia: ArgumentError / AssertionError
    if code == E_NOT_SPD:
        raise NotPositiveDefinite(code, msg)
    if code == E_UNSUPPORTED:
        raise NotImplementedError(msg)
    if code == E_NOMEM:
        raise MemoryError(msg)
    raise LpvsError(code, msg)
