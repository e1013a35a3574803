"""Build libxparcel.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the tree)."""

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(HERE, "libxparcel.so")
CHECK_LIB_PATH = os.path.join(HERE, "libxparcel_check.so")      # -DXP_BOUNDS_CHECK variant (tests only)
SOURCES = ["xp_api.cu", "xp_kernels.cu", "xp_list.cu", "xp_tables.cu", "xp_fast.cu", "xp_derived.cu", "xp_layers.cu", "xp_levels.cu", "xp_downdraft.cu", "xp_effective.cu", "xp_kinematics.cu"]
HEADERS = ["xp_math.cuh", "xp_column.cuh", "xp_parcels.cuh", "xp_kernels.cuh", "xp_fast.cuh", "xp_fast_pcol.cuh", "xp_fast6.cuh", "xp_fast7.cuh", "xp_fast_pcol6.cuh", "xp_fast_pcol7.cuh", "xp_kernels_common.cuh", "xp_layers.cuh", "xp_levels.cuh", "xp_downdraft.cuh", "xp_effective.cuh", "xp_kinematics.cuh",
           os.path.join("..", "..", "include", "xparcel.h")]
NVCC_COMMON = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
               "-Xcompiler", "-fPIC"]
# The float64 exact path must round like the reference's NumPy arithmetic (knife-edge cases such as
# zero-width intervals at a duplicated LCL pressure, PF:1046-1050): no FMA contraction there.  The
# float32 fast path (xp_fast.cu) takes no decision inside its error margin, so it may contract.
PER_FILE_FLAGS = {"xp_fast.cu": [], "xp_api.cu": ["-fmad=false"], "xp_kernels.cu": ["-fmad=false"], "xp_list.cu": ["-fmad=false"],
                  "xp_tables.cu": ["-fmad=false"], "xp_derived.cu": ["-fmad=false"], "xp_layers.cu": ["-fmad=false"],
                  "xp_levels.cu": ["-fmad=false"], "xp_downdraft.cu": ["-fmad=false"],
                  "xp_effective.cu": ["-fmad=false"], "xp_kinematics.cu": ["-fmad=false"]}
LINK_FLAGS = ["-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a"]


def find_nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC or install the CUDA toolkit)")


def is_stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, extra_flags=(), lib_out=None):
    """Compile the CUDA sources into xarray_parcel_b200/libxparcel.so.  Returns the path.
    `extra_flags` / `lib_out` build an experimental variant next to it (A/B runs: XP_LIB_PATH selects it)."""
    if lib_out is None and not force and not is_stale():
        return LIB_PATH
    nvcc = find_nvcc()
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    for src in SOURCES:
        tag = f"{os.getpid()}.{abs(hash((tuple(extra_flags), lib_out))) % 100000}"     # concurrent builds do not collide
        obj = os.path.join(objdir, src.replace(".cu", f".{tag}.o"))
        cmd = [nvcc] + NVCC_COMMON + PER_FILE_FLAGS.get(src, []) + list(extra_flags) + (["-Xptxas", "-v"] if verbose else [])
        cmd += ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)))
    objs, log = [], ""
    for src, obj, pr in procs:
        out, err = pr.communicate()
        log += out + err
        if pr.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n" + out + err)
        objs.append(obj)
    target = lib_out or LIB_PATH
    tmp = target + f".tmp{os.getpid()}"
    res = subprocess.run([nvcc] + LINK_FLAGS + ["-o", tmp] + objs, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc link failed:\n" + res.stdout + res.stderr)
    os.replace(tmp, target)
    for o in objs:
        os.remove(o)
    if verbose:
        print(log)
    return target


if __name__ == "__main__":
    print(build(force=True, verbose=True))
