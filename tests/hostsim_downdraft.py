"""Build and call tests/hostsim/hostsim_downdraft.cpp (TEST-ONLY host compile of xp_downdraft.cuh), built the same way
as tests/hostsim (hostsim_util.py): g++ without FMA contraction, or with XP_HOSTSIM_SANITIZE=1 under ASan + UBSan."""

import ctypes
import os
import subprocess

import numpy as np

import hostsim_util

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "hostsim", "hostsim_downdraft.cpp")
BUILD = os.path.join(HERE, "hostsim", "_build_downdraft_asan" if hostsim_util.SANITIZE else "_build_downdraft")
LIB = os.path.join(BUILD, "libhostsim_downdraft.so")
DEPS = [SRC] + [os.path.join(hostsim_util.CSRC, f) for f in ("xp_math.cuh", "xp_column.cuh", "xp_downdraft.cuh")]


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
        _lib.hostsim_downdraft_cape.restype = None
    return _lib


def _vp(a):
    return ctypes.c_void_p(a.ctypes.data)


def downdraft_cape(p, t, td, tables, metpy_compat=141, profile=False):
    """xp_downdraft.cuh on float64 [L, N] T / Td and pressure [L, N] or a shared [L].  Returns dict of dcape,
    downdraft_start_pressure, downdraft_start_temperature [N], 'levels_read' [N] (1 + the highest level index read)
    and, with ``profile``, downdraft_parcel_temperature [L, N]."""
    t = np.ascontiguousarray(t, dtype=np.float64)
    td = np.ascontiguousarray(td, dtype=np.float64)
    p = np.ascontiguousarray(p, dtype=np.float64)
    L, N = t.shape
    out = np.empty((3, N))
    prof = np.empty((L, N)) if profile else None
    top = np.empty(N, dtype=np.int32)
    idx = np.ascontiguousarray(tables.index_grid, dtype=np.uint16)
    cur = np.ascontiguousarray(tables.curves_asc, dtype=np.float32)
    lib().hostsim_downdraft_cape(_vp(p), int(p.ndim == 1), _vp(t), _vp(td), ctypes.c_int64(N), L, int(metpy_compat),
                                 _vp(idx), _vp(cur), _vp(out), _vp(prof) if profile else None, _vp(top))
    res = {"dcape": out[0], "downdraft_start_pressure": out[1], "downdraft_start_temperature": out[2],
           "levels_read": top}
    if profile:
        res["downdraft_parcel_temperature"] = prof
    return res
