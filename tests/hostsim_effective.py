"""Build and call tests/hostsim/hostsim_effective.cpp (TEST-ONLY host compile of xp_effective.cuh), built the same way
as tests/hostsim (hostsim_util.py): g++ without FMA contraction, or with XP_HOSTSIM_SANITIZE=1 under ASan + UBSan."""

import ctypes
import os
import subprocess

import numpy as np

import hostsim_util

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "hostsim", "hostsim_effective.cpp")
BUILD = os.path.join(HERE, "hostsim", "_build_effective_asan" if hostsim_util.SANITIZE else "_build_effective")
LIB = os.path.join(BUILD, "libhostsim_effective.so")
DEPS = [SRC] + [os.path.join(hostsim_util.CSRC, f)
                for f in ("xp_math.cuh", "xp_column.cuh", "xp_parcels.cuh", "xp_effective.cuh")]


def build():
    if os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(d) for d in DEPS):
        return LIB
    os.makedirs(BUILD, exist_ok=True)
    tmp = LIB + f".tmp{os.getpid()}"
    # -ffp-contract=off: keep host arithmetic un-fused, like NumPy's
    cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-x", "c++", SRC, "-o", tmp]
    if hostsim_util.SANITIZE:
        cmd[1:2] = ["-O1", "-g", "-fsanitize=address,undefined", "-fno-omit-frame-pointer", "-fno-sanitize-recover=undefined"]
    subprocess.run(cmd, check=True)
    os.replace(tmp, LIB)
    return LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
        _lib.hostsim_effective.restype = None
        _lib.hostsim_effective.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                           ctypes.c_int64, ctypes.c_int, ctypes.c_void_p, ctypes.c_double,
                                           ctypes.c_double, ctypes.c_double, ctypes.c_void_p, ctypes.c_void_p,
                                           ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    return _lib


def _vp(a):
    return ctypes.c_void_p(a.ctypes.data)


def effective_inflow_layer(p, t, td, tables, min_cape=100.0, min_cin=-250.0, most_unstable_depth=300.0,
                           virtual_temperature_correction=True, lcl_interp="log", pos_cape_neg_cin=True,
                           post_zero_cin=False, metpy_compat=141):
    """xp_effective.cuh on float64 [L, N] T / Td and pressure [L, N] or a shared [L], in both modes.  Returns a dict
    of base / top [N] of the search mode, all_base / all_top [N] of the all-levels mode, gate [N] (the most-unstable
    parcel passes), level_cape / level_cin [L, N] and flags (search, all-levels)."""
    t = np.ascontiguousarray(t, dtype=np.float64)
    td = np.ascontiguousarray(td, dtype=np.float64)
    p = np.ascontiguousarray(p, dtype=np.float64)
    L, N = t.shape
    out = np.empty((5, N))
    lcape, lcin = np.empty((L, N)), np.empty((L, N))
    flags = np.zeros(2, dtype=np.uint32)
    iopts = np.array([int(bool(virtual_temperature_correction)), int(lcl_interp == "log"), int(bool(pos_cape_neg_cin)),
                      int(bool(post_zero_cin)), int(metpy_compat)], dtype=np.int32)
    idx = np.ascontiguousarray(tables.index_grid, dtype=np.uint16)
    cur = np.ascontiguousarray(tables.curves_asc, dtype=np.float32)
    lib().hostsim_effective(_vp(p), int(p.ndim == 1), _vp(t), _vp(td), N, L, _vp(iopts), float(most_unstable_depth),
                            float(min_cape), float(min_cin), _vp(idx), _vp(cur), _vp(out), _vp(lcape), _vp(lcin),
                            _vp(flags))
    return {"base": out[0], "top": out[1], "all_base": out[2], "all_top": out[3], "gate": out[4] == 1.0, "level_cape": lcape,
            "level_cin": lcin, "flags": (int(flags[0]), int(flags[1]))}
