"""ctypes binding of libhdp_b200.so (the C ABI declared in include/hdp_b200.h).

There is no fallback: if the shared library is missing it is built with nvcc, and if that is impossible
or the library cannot be loaded, every entry point raises.  Nothing in hdp_b200 computes on the CPU.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

from . import build as _build

_i64 = ctypes.c_int64
_int = ctypes.c_int
_p = ctypes.c_void_p
_sz = ctypes.c_size_t

# name -> (restype, argtypes); mirrors include/hdp_b200.h one to one
SIGNATURES = {
    "hdp_b200_abi_version": (_int, []),
    "hdp_b200_strerror": (ctypes.c_char_p, [_int]),
    "hdp_b200_device_info": (_int, [_p, _p, _p]),
    "hdp_b200_launch_count": (_i64, []),
    "hdp_b200_thresholds_workspace_bytes": (_sz, [_i64, _i64, _i64, _i64, _int, _int, _int, _int, _int]),
    "hdp_b200_thresholds": (_int, [_p, _i64, _i64, _i64, _i64, _p, _p, _int, _int, _int, _p, _int, _p, _p, _sz, _p, _int]),
    "hdp_b200_thresholds_force_generic": (None, [_int]),
    "hdp_b200_thresholds_kernel_choice": (_int, [_p, _p, _i64, _int, _int, _int, _p, _int, _p]),
    "hdp_b200_thresholds_host": (_int, [_p, _i64, _i64, _i64, _i64, _p, _p, _int, _int, _int, _p, _int, _p, _p, _int]),
    "hdp_b200_metrics_workspace_bytes": (_sz, [_i64, _i64, _i64, _i64, _int, _int, _int, _int, _p]),
    "hdp_b200_metrics": (_int, [_p, _i64, _i64, _i64, _i64, _p, _int, _int, _p, _p, _int, _p, _p, _int, _p, _p, _p, _sz, _p, _int]),
    "hdp_b200_metrics_host": (_int, [_p, _i64, _i64, _i64, _i64, _p, _p, _int, _int, _p, _p, _int, _p, _p, _int, _p, _p, _int]),
    "hdp_b200_intensity_workspace_bytes": (_sz, [_i64, _i64, _i64, _i64, _int, _int, _int, _int, _p]),
    "hdp_b200_intensity": (_int, [_p, _i64, _i64, _i64, _i64, _p, _int, _int, _p, _p, _int, _p, _p, _int, _p, _p, _p, _p, _sz, _p, _int]),
    "hdp_b200_intensity_host": (_int, [_p, _i64, _i64, _i64, _i64, _p, _p, _int, _int, _p, _p, _int, _p, _p, _int, _p, _p, _p, _int]),
    "hdp_b200_compound_workspace_bytes": (_sz, [_i64, _i64, _i64, _i64, _int, _int, _int, _int, _p]),
    "hdp_b200_compound": (_int, [_p, _i64, _i64, _p, _i64, _i64, _i64, _i64, _p, _p, _int, _int, _p, _p, _int, _p, _p, _int, _p, _p, _p,
                                 _p, _sz, _p, _int]),
    "hdp_b200_compound_host": (_int, [_p, _i64, _i64, _p, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _int, _int, _p, _p, _int, _p, _p, _int,
                                      _p, _p, _p, _int]),
    "hdp_b200_compound_hot_days": (_int, [_p, _i64, _i64, _p, _i64, _i64, _i64, _i64, _p, _p, _int, _int, _p, _p, _p, _sz, _p, _int]),
    "hdp_b200_compound_plan": (_int, [_int, _p]),
    "hdp_b200_host_release": (None, []),
    "hdp_b200_metrics_run_filter": (None, [_int]),
    "hdp_b200_metrics_kernel_choice": (_int, [_p, _int, _p, _p, _int, _i64, _p]),
    "hdp_b200_heat_index": (_int, [_p, _p, _i64, _p, _p]),
    "hdp_b200_heat_index_measure": (_int, [_p, _p, _i64, _int, _p, _p]),
    "hdp_b200_to_celsius": (_int, [_p, _i64, _int, _p, _p]),
    "hdp_b200_weighted_mean": (_int, [_p, _i64, _i64, _p, ctypes.c_double, _p, _p]),
    "hdp_b200_timing_enable": (None, [_int]),
    "hdp_b200_timing_read": (_int, [_p, _p, _int]),
    "hdp_b200_hot_days": (_int, [_p, _i64, _i64, _i64, _i64, _p, _int, _int, _p, _p, _p, _sz, _p]),
    "hdp_b200_index_heatwaves": (_int, [_p, _i64, _i64, _p, _int, _p, _p]),
    "hdp_b200_season_metrics": (_int, [_p, _i64, _i64, _p, _int, _p, _p, _p, _p, _p]),
}

_LIB: Optional[ctypes.CDLL] = None


class HdpB200Error(RuntimeError):
    def __init__(self, code: int, where: str):
        self.code = code
        msg = lib().hdp_b200_strerror(code).decode()
        super().__init__(f"{where} failed with code {code}: {msg}")


def lib_path() -> str:
    return _build.LIB


def lib() -> ctypes.CDLL:
    """Load (building first if needed) libhdp_b200.so.  Raises if that is not possible."""
    global _LIB
    if _LIB is None:
        path = _build.LIB
        if not os.path.exists(path) or (os.path.isdir(_build.CSRC) and not _build.up_to_date() and _can_build()):
            path = _build.build()
        L = ctypes.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)          # AttributeError if the library does not export the symbol
            fn.restype = res
            fn.argtypes = args
        if L.hdp_b200_abi_version() != 6:
            raise RuntimeError("libhdp_b200.so ABI version mismatch; rebuild with `python -m hdp_b200.build --force`")
        _LIB = L
    return _LIB


def _can_build() -> bool:
    try:
        _build.nvcc()
        return True
    except RuntimeError:
        return False


def check(code: int, where: str) -> None:
    if code != 0:
        raise HdpB200Error(code, where)
