"""Loader for the in-tree CUDA library ``libwva_b200.so`` (C ABI of include/wva_b200.h).

There is no CPU fallback: if the library is missing the import of anything that needs it
raises, and ``Engine()`` raises when no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

from . import _abi

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libwva_b200.so")
SOURCES = [os.path.join(_HERE, "csrc", n) for n in ("wva_b200.cu", "wva_kernels.cuh", "wva_device.cuh", "wva_size.cuh")]
HEADER = os.path.join(os.path.dirname(_HERE), "include", "wva_b200.h")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false",  # the reference never contracts a*b+c (Go/amd64); explicit __fma_rn only
    "-shared", "-Xcompiler", "-fPIC",
]


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile the CUDA library for sm_100a in-tree (cross-compiles without a GPU)."""
    deps = SOURCES + [HEADER]
    stale = (not os.path.exists(SO_PATH)) or any(os.path.getmtime(p) > os.path.getmtime(SO_PATH) for p in deps)
    if force or stale:
        nvcc = os.environ.get("NVCC", "nvcc")
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", SO_PATH, SOURCES[0]]
        subprocess.run(cmd, check=True)
    return SO_PATH


EXPORTS = (
    "wva_tunables_default", "wva_create", "wva_destroy", "wva_strerror", "wva_last_error", "wva_abi_version",
    "wva_analyze", "wva_solve", "wva_grid_solve", "wva_sweep", "wva_upload", "wva_update_load", "wva_resolve",
    "wva_grid_solve_device", "wva_resolve_device", "wva_stream", "wva_synchronize", "wva_launch_count",
    "wva_last_kernel_ms", "wva_last_device_ms", "wva_summarize", "wva_solve_greedy", "wva_mm1k_solve",
    "wva_xchg_create", "wva_xchg_open", "wva_xchg_publish", "wva_xchg_error", "wva_xchg_destroy",
    "wva_resolve_scenarios",
)

_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise RuntimeError(f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback for the CUDA path)")
    L = C.CDLL(SO_PATH)
    vp, i32, f32p, i32p = C.c_void_p, C.c_int32, _abi.f32p, _abi.i32p
    L.wva_tunables_default.argtypes = [C.POINTER(_abi.Tunables)]
    L.wva_create.restype = C.c_int
    L.wva_create.argtypes = [C.POINTER(vp), C.c_int]
    L.wva_destroy.argtypes = [vp]
    L.wva_strerror.restype = C.c_char_p
    L.wva_strerror.argtypes = [C.c_int]
    L.wva_last_error.restype = C.c_char_p
    L.wva_last_error.argtypes = [vp]
    L.wva_abi_version.restype = C.c_int
    for name, args in (
        ("wva_analyze", [vp, C.POINTER(_abi.FleetC), C.POINTER(_abi.AllocsC)]),
        ("wva_solve", [vp, C.POINTER(_abi.FleetC), C.POINTER(_abi.AllocsC), C.POINTER(_abi.AllocsC)]),
        ("wva_grid_solve", [vp, C.POINTER(_abi.FleetC), C.POINTER(_abi.GridC), C.POINTER(_abi.CellsC),
                            C.POINTER(_abi.AllocsC)]),
        ("wva_sweep", [vp, C.POINTER(_abi.FleetC), i32, C.POINTER(_abi.SweepOutC)]),
        ("wva_upload", [vp, C.POINTER(_abi.FleetC)]),
        ("wva_update_load", [vp, f32p, i32p, i32p]),
        ("wva_resolve", [vp, C.POINTER(_abi.AllocsC), C.POINTER(_abi.AllocsC)]),
        ("wva_resolve_scenarios", [vp, i32, f32p, C.POINTER(_abi.AllocsC), C.POINTER(_abi.AllocsC)]),
        ("wva_grid_solve_device", [vp, C.POINTER(_abi.GridC), C.POINTER(_abi.AllocsC)]),
        ("wva_resolve_device", [vp, C.POINTER(_abi.AllocsC)]),
        ("wva_synchronize", [vp]),
        ("wva_solve_greedy", [C.POINTER(_abi.FleetC), C.POINTER(_abi.AllocsC), C.POINTER(_abi.AllocsC)]),
        ("wva_summarize", [vp, C.POINTER(_abi.SummaryC)]),
        ("wva_mm1k_solve", [vp, i32, i32p, f32p, f32p, C.POINTER(_abi.Mm1kOutC)]),
        ("wva_xchg_create", [vp, C.c_int, C.c_int, C.c_size_t, C.c_void_p]),
        ("wva_xchg_open", [vp, C.c_int, C.c_void_p]),
        ("wva_xchg_publish", [vp, C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
        ("wva_xchg_error", [vp]),
        ("wva_xchg_destroy", [vp]),
    ):
        fn = getattr(L, name)
        fn.restype = C.c_int
        fn.argtypes = args
    L.wva_stream.restype = vp
    L.wva_stream.argtypes = [vp]
    L.wva_launch_count.restype = C.c_int64
    L.wva_launch_count.argtypes = [vp]
    L.wva_last_kernel_ms.restype = C.c_float
    L.wva_last_kernel_ms.argtypes = [vp]
    L.wva_last_device_ms.restype = C.c_float
    L.wva_last_device_ms.argtypes = [vp]
    _lib = L
    return L
