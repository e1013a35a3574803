"""Build and call tests/hostsim/hostsim_kinematics.cpp (TEST-ONLY host compile of xp_kinematics.cuh), built the same
way as tests/hostsim (hostsim_util.py): g++ without FMA contraction, or with XP_HOSTSIM_SANITIZE=1 under ASan + UBSan."""

import ctypes
import os
import subprocess

import numpy as np

import hostsim_util

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "hostsim", "hostsim_kinematics.cpp")
BUILD = os.path.join(HERE, "hostsim", "_build_kinematics_asan" if hostsim_util.SANITIZE else "_build_kinematics")
LIB = os.path.join(BUILD, "libhostsim_kinematics.so")
DEPS = [SRC] + [os.path.join(hostsim_util.CSRC, f) for f in ("xp_math.cuh", "xp_kinematics.cuh")]

OUT_FIELDS = ["bunkers_right_u", "bunkers_right_v", "bunkers_left_u", "bunkers_left_v", "mean_wind_u", "mean_wind_v",
              "srh0", "srh1", "srh2", "srh3", "srh_layer", "bulk_wind_difference_u", "bulk_wind_difference_v",
              "bulk_wind_difference"]


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
        _lib.hostsim_storm_kinematics.restype = None
        _lib.hostsim_storm_kinematics.argtypes = [ctypes.c_void_p] * 5 + [ctypes.c_int64] + [ctypes.c_int] * 4 + \
            [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        _lib.hostsim_composites.restype = None
        _lib.hostsim_composites.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]
    return _lib


def _vp(a):
    return ctypes.c_void_p(a.ctypes.data)


def storm_kinematics(z, u, v, su, sv, mover=1, depths=(), srh_layer=None, bwd_layer=None, motion=True):
    """xp_kinematics.cuh on float64 [L, N] height / winds and [N] surface winds.  Returns a dict with the names of
    kinematics_oracle.storm_kinematics plus 'levels_read' [N] (1 + the highest level index read)."""
    z, u, v = [np.ascontiguousarray(x, dtype=np.float64) for x in (z, u, v)]
    L, N = z.shape
    su, sv = [np.ascontiguousarray(np.broadcast_to(np.asarray(x, np.float64), (N,))) for x in (su, sv)]
    layers = np.full((4, N), np.nan)
    if srh_layer is not None:
        layers[0], layers[1] = srh_layer
    if bwd_layer is not None:
        layers[2], layers[3] = bwd_layer
    d = np.zeros(4)
    d[:len(depths)] = depths
    out = np.empty((len(OUT_FIELDS), N))
    top = np.empty(N, dtype=np.int32)
    lib().hostsim_storm_kinematics(_vp(z), _vp(u), _vp(v), _vp(su), _vp(sv), N, L, int(motion), int(mover),
                                   len(depths), _vp(d), int(srh_layer is not None), int(bwd_layer is not None),
                                   _vp(layers), _vp(out), _vp(top))
    res = {k: out[i] for i, k in enumerate(OUT_FIELDS) if not k.startswith("srh")}
    for j, dd in enumerate(depths):
        res[f"srh_0_{float(dd):g}m"] = out[6 + j]
    if srh_layer is not None:
        res["srh_layer"] = out[10]
    if bwd_layer is None:
        for k in ("bulk_wind_difference_u", "bulk_wind_difference_v", "bulk_wind_difference"):
            del res[k]
    res["levels_read"] = top
    return res


def composites(mucape, esrh, ebwd, mlcape, mlcin, lcl_height):
    """(scp, stp) of xp_kinematics.cuh on broadcast float64 inputs."""
    xs = np.broadcast_arrays(*[np.asarray(x, np.float64) for x in (mucape, esrh, ebwd, mlcape, mlcin, lcl_height)])
    shape = xs[0].shape
    inp = np.ascontiguousarray(np.stack([x.ravel() for x in xs]))
    n = inp.shape[1]
    out = np.empty((2, n))
    lib().hostsim_composites(_vp(inp), n, _vp(out))
    return out[0].reshape(shape), out[1].reshape(shape)
