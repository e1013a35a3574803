"""ctypes binding of libxparcel.so (the C ABI declared in include/xparcel.h).

This is the binding a maintainer of the reference would add (INTEGRATION.md).  PyTorch is
used only for device/pinned memory and streams; no torch type crosses the ABI -- only raw
pointers, sizes and a cudaStream_t.
"""

import ctypes
import os
import threading

import torch

from . import _build

c_void_p, c_int32, c_int64, c_double = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_double

XP_OK = 0
XP_F32, XP_F64 = 0, 1
XP_MEM_DEVICE, XP_MEM_HOST = 0, 1
KIND = {"sb": 0, "ml": 1, "mu": 2, "explicit": 3}
FLAG_TOP_TEMPERATURE_NAN = 1
FLAG_PRESSURES_NOT_UNIQUE = 2
FLAG_PRESSURE_NOT_DECREASING = 4
FLAG_PRESSURE_ORDER_CHECKED = 8
TABLE_NP, TABLE_NT, TABLE_NADIABATS = 2196, 7150, 14300

SCALAR_FIELDS = ["cape", "cin", "lcl_pressure", "lcl_temperature", "lcl_virtual_temperature",
                 "lfc_pressure", "lfc_temperature", "el_pressure", "el_temperature",
                 "parcel_pressure", "parcel_temperature", "parcel_dewpoint"]
PROFILE_FIELDS = ["profile_pressure", "profile_temperature", "profile_virtual_temperature",
                  "profile_environment_temperature", "profile_environment_virtual_temperature",
                  "profile_environment_dewpoint"]


class XpColumns(ctypes.Structure):
    _fields_ = [("pressure", c_void_p), ("temperature", c_void_p), ("dewpoint", c_void_p),
                ("n_columns", c_int64), ("n_levels", c_int32), ("dtype", c_int32),
                ("level_stride", c_int64), ("pressure_level_stride", c_int64),
                ("pressure_is_1d", c_int32), ("mem", c_int32),
                ("dewpoint_is_specific_humidity", c_int32), ("reserved_", c_int32)]


class XpOptions(ctypes.Structure):
    _fields_ = [("virtual_temperature_correction", c_int32), ("lcl_interp_log", c_int32),
                ("pos_cape_neg_cin", c_int32), ("post_zero_cin", c_int32),
                ("metpy_compat", c_int32), ("exact_only", c_int32),
                ("mixed_layer_depth", c_double), ("most_unstable_depth", c_double)]


class XpParcelOut(ctypes.Structure):
    _fields_ = ([(f, c_void_p) for f in SCALAR_FIELDS] + [("level_shift", c_void_p)] +
                [(f, c_void_p) for f in PROFILE_FIELDS] + [("profile_level_stride", c_int64)])


class XpParcelIn(ctypes.Structure):
    _fields_ = [("pressure", c_void_p), ("temperature", c_void_p), ("dewpoint", c_void_p)]


EXPORTS = ["xp_version", "xp_create", "xp_destroy", "xp_last_error", "xp_take_flags",
           "xp_default_options", "xp_tables_build", "xp_tables_set", "xp_tables_get",
           "xp_tables_loaded", "xp_cape_cin", "xp_suite", "xp_lcl", "xp_moist_lapse",
           "xp_parcel_profile", "xp_lfc_el", "xp_cape_cin_base", "xp_launch_count",
           "xp_last_kernel_ms", "xp_last_kernel_split_ms", "xp_last_exact_count", "xp_interp_levels",
           "xp_level_crossing", "xp_dewpoint_from_specific_humidity", "xp_saturation_mixing_ratio",
           "xp_dry_lapse", "xp_mixing_ratio", "xp_virtual_temperature", "xp_wet_bulb_temperature",
           "xp_significant_hail_parameter", "xp_storm_proxies", "xp_mixed_layer", "xp_mixed_parcel",
           "xp_layer_bounds", "xp_insert_level", "xp_shift_out_nans", "xp_trapz", "xp_valid_data",
           "xp_find_intersections", "xp_interp1d", "xp_trap_around_zeros", "xp_downdraft_cape",
           "xp_effective_inflow_layer"]

PROXY_INPUTS = ["mixed_100_cape", "mixed_50_cape", "mu_cape", "shear_magnitude", "mixed_100_lifted_index",
                "mixed_100_dci", "positive_shear", "mixed_50_cin", "mixed_100_cin", "lapse_rate_700_500",
                "mu_mixing_ratio", "temp_500", "freezing_level"]
PROXY_FLAGS = ["proxy_Craven2004", "proxy_Kunz2007", "proxy_Trapp2007", "proxy_Marsh2009", "proxy_Allen2011",
               "proxy_Allen2014", "proxy_Eccel2012", "proxy_Mohr2013", "proxy_SHIP_0.1"]


MIXED_PARCEL_FIELDS = ["theta", "mixing_ratio", "temperature", "vapour_pressure", "dewpoint", "pressure"]


class XpMixedParcelOut(ctypes.Structure):
    _fields_ = [(n, c_void_p) for n in MIXED_PARCEL_FIELDS]


INTERSECTION_FIELDS = ["all_intersect_x", "all_intersect_y", "increasing_x", "increasing_y", "decreasing_x",
                       "decreasing_y"]


class XpIntersectionsOut(ctypes.Structure):
    _fields_ = [(n, c_void_p) for n in INTERSECTION_FIELDS]


ZERO_AREA_FIELDS = ["area", "x", "dx", "x_from", "x_to"]


class XpZeroAreasOut(ctypes.Structure):
    _fields_ = [(n, c_void_p) for n in ZERO_AREA_FIELDS] + [("mask", c_void_p)]


DOWNDRAFT_FIELDS = ["dcape", "downdraft_start_pressure", "downdraft_start_temperature"]


class XpDowndraftOut(ctypes.Structure):
    _fields_ = [("dcape", c_void_p), ("start_pressure", c_void_p), ("start_temperature", c_void_p),
                ("parcel_temperature", c_void_p), ("parcel_level_stride", c_int64)]


EFFECTIVE_FIELDS = ["effective_inflow_base", "effective_inflow_top"]
EFFECTIVE_LEVEL_FIELDS = ["level_parcel_cape", "level_parcel_cin"]


class XpEffectiveOut(ctypes.Structure):
    _fields_ = [("base_pressure", c_void_p), ("top_pressure", c_void_p), ("level_cape", c_void_p),
                ("level_cin", c_void_p), ("level_out_stride", c_int64)]


class XpProxyInputs(ctypes.Structure):
    _fields_ = [(n, c_void_p) for n in PROXY_INPUTS]


class XpProxyOutputs(ctypes.Structure):
    _fields_ = [(f"flag{i}", c_void_p) for i in range(9)] + [("ship", c_void_p)]


class XparcelError(RuntimeError):
    pass


_lib = None
_lib_lock = threading.Lock()


def load_library():
    """dlopen xarray_parcel_b200/libxparcel.so.  There is no fallback: a missing library is an
    error (build it with ``python -m xarray_parcel_b200._build`` / ``__graft_entry__.build()``)."""
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        path = os.environ.get("XP_LIB_PATH") or _build.LIB_PATH      # XP_LIB_PATH: an experimental build (A/B runs)
        if not os.path.exists(path):
            raise XparcelError(f"{path} is missing: build the CUDA library first "
                               "(python -m xarray_parcel_b200._build); there is no CPU fallback")
        lib = ctypes.CDLL(path)
        lib.xp_version.restype = ctypes.c_char_p
        lib.xp_last_error.restype = ctypes.c_char_p
        lib.xp_last_error.argtypes = [c_void_p]
        lib.xp_create.argtypes = [ctypes.c_int, ctypes.POINTER(c_void_p)]
        lib.xp_destroy.argtypes = [c_void_p]
        lib.xp_destroy.restype = None
        lib.xp_take_flags.argtypes = [c_void_p, c_void_p, ctypes.POINTER(ctypes.c_uint32)]
        lib.xp_default_options.argtypes = [ctypes.POINTER(XpOptions)]
        lib.xp_default_options.restype = None
        lib.xp_tables_build.argtypes = [c_void_p, c_void_p]
        lib.xp_tables_set.argtypes = [c_void_p, c_void_p, c_void_p]
        lib.xp_tables_get.argtypes = [c_void_p, c_void_p, c_void_p]
        lib.xp_tables_loaded.argtypes = [c_void_p]
        lib.xp_cape_cin.argtypes = [c_void_p, ctypes.POINTER(XpColumns), c_int32,
                                    ctypes.POINTER(XpParcelIn), ctypes.POINTER(XpOptions),
                                    ctypes.POINTER(XpParcelOut), c_void_p]
        lib.xp_suite.argtypes = [c_void_p, ctypes.POINTER(XpColumns), ctypes.POINTER(XpOptions),
                                 ctypes.POINTER(XpParcelOut), ctypes.POINTER(XpParcelOut),
                                 ctypes.POINTER(XpParcelOut), c_void_p]
        lib.xp_lcl.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32,
                               ctypes.POINTER(XpOptions), c_void_p, c_void_p, c_void_p, c_void_p]
        lib.xp_moist_lapse.argtypes = [c_void_p, c_void_p, c_int64, c_int32, c_int64, c_int32,
                                       c_void_p, c_void_p, c_void_p, c_int64, c_void_p]
        lib.xp_parcel_profile.argtypes = [c_void_p, c_void_p, c_int64, c_int32, c_int64, c_int32,
                                          ctypes.POINTER(XpParcelIn), ctypes.POINTER(XpOptions),
                                          c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                                          c_void_p]
        lib.xp_lfc_el.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int64,
                                  c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_void_p]
        lib.xp_cape_cin_base.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32,
                                         c_int64, c_int32, c_void_p, c_void_p,
                                         ctypes.POINTER(XpOptions), c_void_p, c_void_p, c_void_p]
        lib.xp_interp_levels.argtypes = [c_void_p, c_void_p, c_int64, c_int32, ctypes.POINTER(c_void_p),
                                         ctypes.POINTER(c_void_p), c_int32, c_int64, c_int32, c_int64, c_int32,
                                         c_void_p, c_double, c_int32, c_void_p]
        lib.xp_level_crossing.argtypes = [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_int64, c_int32,
                                          c_int64, c_int32, c_double, c_void_p, c_void_p]
        lib.xp_dewpoint_from_specific_humidity.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32,
                                                           c_int32, c_void_p, c_void_p]
        lib.xp_saturation_mixing_ratio.argtypes = [c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p]
        lib.xp_dry_lapse.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p]
        lib.xp_mixing_ratio.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_void_p,
                                        c_void_p]
        lib.xp_virtual_temperature.argtypes = [c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_double, c_void_p,
                                               c_void_p]
        lib.xp_wet_bulb_temperature.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_void_p,
                                                c_void_p]
        lib.xp_significant_hail_parameter.argtypes = [c_void_p] + [c_void_p] * 6 + [c_int64, c_int32, c_void_p, c_void_p]
        lib.xp_storm_proxies.argtypes = [c_void_p, ctypes.POINTER(XpProxyInputs), c_int64, c_int32,
                                         ctypes.POINTER(XpProxyOutputs), c_void_p]
        lib.xp_mixed_layer.argtypes = [c_void_p, c_void_p, c_int64, c_int32, ctypes.POINTER(c_void_p),
                                       ctypes.POINTER(c_void_p), c_int32, c_int32, c_int64, c_int32, c_int64,
                                       c_int32, c_double, c_void_p]
        lib.xp_mixed_parcel.argtypes = [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_int64, c_int32,
                                        c_int64, c_int32, c_double, ctypes.POINTER(XpMixedParcelOut), c_void_p]
        lib.xp_layer_bounds.argtypes = [c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int64, c_int32, c_double,
                                        c_int32, c_void_p, c_void_p, c_void_p]
        PP = ctypes.POINTER(c_void_p)
        lib.xp_insert_level.argtypes = [c_void_p, c_void_p, c_int64, c_int32, c_void_p, PP, PP, PP, c_int32, c_void_p,
                                        c_int64, c_int64, c_int32, c_int64, c_int32, c_void_p]
        lib.xp_shift_out_nans.argtypes = [c_void_p, c_void_p, PP, PP, c_int32, c_int64, c_int32, c_int64, c_int32,
                                          c_void_p, c_void_p]
        lib.xp_trapz.argtypes = [c_void_p, c_void_p, c_int64, c_int32, PP, PP, c_int32, c_int64, c_int32, c_int64,
                                 c_int32, c_void_p, c_int64, c_int32, c_void_p]
        lib.xp_valid_data.argtypes = [c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int64, c_int32, c_void_p]
        lib.xp_find_intersections.argtypes = [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_int64, c_int64,
                                              c_int32, c_int64, c_int32, c_int32, ctypes.POINTER(XpIntersectionsOut),
                                              c_void_p]
        lib.xp_interp1d.argtypes = [c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_int64, c_int32, c_int32,
                                    c_int32, c_void_p]
        lib.xp_trap_around_zeros.argtypes = [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_int64, c_int64, c_int32,
                                             c_int64, c_int32, c_int32, ctypes.POINTER(XpZeroAreasOut), c_void_p]
        lib.xp_downdraft_cape.argtypes = [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_int64, c_int32,
                                          c_int64, c_int32, c_int32, ctypes.POINTER(XpDowndraftOut), c_void_p]
        lib.xp_effective_inflow_layer.argtypes = [c_void_p, ctypes.POINTER(XpColumns), ctypes.POINTER(XpOptions),
                                                  c_double, c_double, ctypes.POINTER(XpEffectiveOut), c_void_p]
        lib.xp_launch_count.argtypes = [c_void_p]
        lib.xp_launch_count.restype = ctypes.c_uint64
        lib.xp_last_kernel_ms.argtypes = [c_void_p, ctypes.POINTER(ctypes.c_float)]
        lib.xp_last_kernel_split_ms.argtypes = [c_void_p, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float)]
        lib.xp_last_exact_count.argtypes = [c_void_p, ctypes.POINTER(c_int64)]
        _lib = lib
        return lib


def make_options(virtual_temperature_correction=True, lcl_interp="log", pos_cape_neg_cin=True,
                 post_zero_cin=False, metpy_compat="1.4.1", mixed_layer_depth=100.0,
                 most_unstable_depth=300.0, exact_only=False):
    assert lcl_interp in ["linear", "log"], "interpolator must be linear or log"   # PF:878
    compat = {"1.4.1": 141, "1.6.2": 162, 141: 141, 162: 162}[metpy_compat]
    return XpOptions(int(bool(virtual_temperature_correction)), int(lcl_interp == "log"),
                     int(bool(pos_cape_neg_cin)), int(bool(post_zero_cin)), compat, int(bool(exact_only)),
                     float(mixed_layer_depth), float(most_unstable_depth))


def _dtype_code(t):
    if t.dtype == torch.float32:
        return XP_F32
    if t.dtype == torch.float64:
        return XP_F64
    raise TypeError(f"unsupported dtype {t.dtype}: float32 or float64 required")


class Context:
    """One xp_context (tables + staging) on one CUDA device."""

    def __init__(self, device=0):
        self.lib = load_library()
        if not torch.cuda.is_available():
            raise XparcelError("no CUDA device available: xarray_parcel_b200 has no CPU fallback")
        self.device = int(device)
        h = c_void_p()
        st = self.lib.xp_create(self.device, ctypes.byref(h))
        if st != XP_OK:
            raise XparcelError(f"xp_create failed ({st}): {self.lib.xp_last_error(None).decode()}")
        self.handle = h

    def close(self):
        if getattr(self, "handle", None):
            self.lib.xp_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, st, what):
        if st != XP_OK:
            msg = self.lib.xp_last_error(self.handle).decode()
            if st == 3:
                raise AssertionError(msg)          # PF:60-61
            raise XparcelError(f"{what} failed ({st}): {msg}")

    def _stream(self):
        return c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- tables -------------------------------------------------------------------------
    def tables_loaded(self):
        return bool(self.lib.xp_tables_loaded(self.handle))

    def tables_build(self):
        self._check(self.lib.xp_tables_build(self.handle, self._stream()), "xp_tables_build")

    def tables_set(self, index_grid, curves):
        import numpy as np
        idx = np.ascontiguousarray(index_grid, dtype=np.uint16)
        cur = np.ascontiguousarray(curves, dtype=np.float32)
        assert idx.shape == (TABLE_NP, TABLE_NT) and cur.shape == (TABLE_NADIABATS, TABLE_NP)
        self._check(self.lib.xp_tables_set(self.handle, idx.ctypes.data, cur.ctypes.data), "xp_tables_set")

    def tables_get(self):
        import numpy as np
        idx = np.empty((TABLE_NP, TABLE_NT), dtype=np.uint16)
        cur = np.empty((TABLE_NADIABATS, TABLE_NP), dtype=np.float32)
        self._check(self.lib.xp_tables_get(self.handle, idx.ctypes.data, cur.ctypes.data), "xp_tables_get")
        return idx, cur

    def take_flags(self):
        f = ctypes.c_uint32(0)
        self._check(self.lib.xp_take_flags(self.handle, self._stream(), ctypes.byref(f)), "xp_take_flags")
        return f.value

    def launch_count(self):
        return int(self.lib.xp_launch_count(self.handle))

    def last_exact_count(self):
        """Columns of the last call that the float32 fast path handed to the exact kernel (-1: the
        call did not use the fast path).  For a call on CPU tensors (host memory, staged through the device in
        column blocks of XP_HOST_BLOCK_MB on XP_HOST_THREADS copy threads): the sum over all its blocks (-1: no
        block took the fast path)."""
        n = c_int64(0)
        self._check(self.lib.xp_last_exact_count(self.handle, ctypes.byref(n)), "xp_last_exact_count")
        return n.value

    def last_kernel_ms(self):
        ms = ctypes.c_float(0)
        self._check(self.lib.xp_last_kernel_ms(self.handle, ctypes.byref(ms)), "xp_last_kernel_ms")
        return ms.value

    def last_kernel_split_ms(self):
        """(sweep ms, fix-up ms) of the most recent timed fast-path call (xp_last_kernel_split_ms)."""
        a, b = ctypes.c_float(0), ctypes.c_float(0)
        self._check(self.lib.xp_last_kernel_split_ms(self.handle, ctypes.byref(a), ctypes.byref(b)),
                    "xp_last_kernel_split_ms")
        return a.value, b.value

    # ---- fused path -----------------------------------------------------------------------
    def _columns(self, p, t, td):
        if t.dim() != 2 or td.shape != t.shape:
            raise ValueError("temperature/dewpoint must be [n_levels, n_columns]")
        L, N = t.shape
        if t.dtype != td.dtype or t.dtype != p.dtype:
            raise TypeError("pressure, temperature and dewpoint must share a dtype")
        if t.device != td.device or t.device != p.device:
            raise ValueError("pressure, temperature and dewpoint must be on one device")
        if N > 1 and (t.stride(1) != 1 or td.stride(1) != 1):
            raise ValueError("columns must be contiguous (level-major layout)")
        if t.stride(0) != td.stride(0):
            raise ValueError("temperature and dewpoint must share their level stride")
        p1d = p.dim() == 1
        if p1d:
            if p.shape[0] != L:
                raise ValueError("1-D pressure must have n_levels entries")
            pls = p.stride(0) if L > 1 else 1
        else:
            if p.shape != t.shape or (N > 1 and p.stride(1) != 1):
                raise ValueError("pressure must be [n_levels] or level-major [n_levels, n_columns]")
            pls = p.stride(0) if L > 1 else N
        mem = XP_MEM_DEVICE if t.is_cuda else XP_MEM_HOST
        if t.is_cuda and t.device.index != self.device:
            raise ValueError(f"tensors are on {t.device}, context is on cuda:{self.device}")
        ls = t.stride(0) if L > 1 else N
        # a broadcast view (stride 0 along the levels, e.g. t.expand(L, N)) would make the kernels read L*N
        # elements of an N-element allocation: reject it instead of inventing a stride
        if L > 1 and ls < N:
            raise ValueError("temperature/dewpoint level stride is smaller than n_columns "
                             "(broadcast or overlapping view): call .contiguous() first")
        if not p1d and L > 1 and pls < N:
            raise ValueError("pressure level stride is smaller than n_columns "
                             "(broadcast or overlapping view): call .contiguous() first")
        if p1d and L > 1 and pls < 1:
            raise ValueError("1-D pressure must not be a broadcast view")
        return XpColumns(p.data_ptr(), t.data_ptr(), td.data_ptr(), N, L, _dtype_code(t),
                         ls, pls, int(p1d), mem), L, N

    def _alloc_out(self, like, N, L, profile, pin, fields=None, shift=True):
        """Output block for one parcel kind: scalars [n_fields, N], shift [N], optional profile
        [6, L+1, N].  ``fields`` restricts the scalar outputs (NULL pointers are not written)."""
        kw = dict(dtype=like.dtype, device=like.device)
        pin = pin and not like.is_cuda
        names = list(SCALAR_FIELDS) if fields is None else [f for f in SCALAR_FIELDS if f in fields]
        scal = torch.empty((len(names), N), pin_memory=pin, **kw)
        sh = torch.empty((N,), dtype=torch.int32, device=like.device, pin_memory=pin) if shift else None
        prof = torch.empty((len(PROFILE_FIELDS), L + 1, N), pin_memory=pin, **kw) if profile else None
        po = XpParcelOut()
        for i, f in enumerate(names):
            setattr(po, f, scal[i].data_ptr())
        if sh is not None:
            po.level_shift = sh.data_ptr()
        if prof is not None:
            for i, f in enumerate(PROFILE_FIELDS):
                setattr(po, f, prof[i].data_ptr())
        po.profile_level_stride = N
        return po, scal, sh, prof, names

    def alloc_outputs(self, like, kinds=("sb",), profile=False, pin_outputs=False, fields=None,
                      shift=True):
        """Reusable output blocks for ``cape_cin(..., out=...)`` (``like``: the temperature block
        [L, N]).  ``fields`` may be a list (all kinds) or {kind: list}."""
        L, N = like.shape
        outs = {}
        for k in kinds:
            f = fields.get(k) if isinstance(fields, dict) else fields
            outs[k] = self._alloc_out(like, N, L, profile, pin_outputs, f, shift)
        return outs

    def output_bytes(self, outs):
        """Bytes the library writes into an ``alloc_outputs`` block set."""
        n = 0
        for po, scal, sh, prof, _ in outs.values():
            n += scal.numel() * scal.element_size()
            n += sh.numel() * 4 if sh is not None else 0
            n += prof.numel() * prof.element_size() if prof is not None else 0
        return n

    def cape_cin(self, p, t, td, kinds=("sb",), options=None, profile=False, explicit=None,
                 pin_outputs=False, out=None, specific_humidity=False):
        """Run the fused kernel for the requested parcel kinds on level-major torch tensors.

        CUDA tensors: asynchronous on the current stream.  CPU tensors: staged through the
        device by the library (host path of the C ABI).  Returns {kind: {field: tensor}}.
        ``specific_humidity=True``: ``td`` holds specific humidity [kg/kg]; the kernels convert it to the dewpoint
        as each level is loaded (metpy.calc.dewpoint_from_specific_humidity in the options' metpy_compat form,
        PF:1889, 1969) -- no dewpoint array is materialised.
        """
        opts = options if options is not None else make_options()
        cols, L, N = self._columns(p, t, td)
        cols.dewpoint_is_specific_humidity = int(bool(specific_humidity))
        kinds = tuple(kinds)
        keep = {}
        outs = out if out is not None else self.alloc_outputs(t, kinds, profile, pin_outputs)
        if set(kinds) <= {"sb", "ml", "mu"} and len(kinds) > 1:
            ptrs = [ctypes.byref(outs[k][0]) if k in kinds else None for k in ("sb", "ml", "mu")]
            st = self.lib.xp_suite(self.handle, ctypes.byref(cols), ctypes.byref(opts), ptrs[0], ptrs[1],
                                   ptrs[2], self._stream())
            self._check(st, "xp_suite")
        else:
            for k in kinds:
                pin = None
                if k == "explicit":
                    ep, et, etd = [e.contiguous() for e in explicit]
                    keep[k] = (ep, et, etd)
                    pin = ctypes.byref(XpParcelIn(ep.data_ptr(), et.data_ptr(), etd.data_ptr()))
                st = self.lib.xp_cape_cin(self.handle, ctypes.byref(cols), KIND[k], pin,
                                          ctypes.byref(opts), ctypes.byref(outs[k][0]), self._stream())
                self._check(st, "xp_cape_cin")
        res = {}
        for k in kinds:
            _, scal, shift, prof, names = outs[k]
            d = {f: scal[i] for i, f in enumerate(names)}
            if shift is not None:
                d["level_shift"] = shift
            if prof is not None:
                for i, f in enumerate(PROFILE_FIELDS):
                    d[f] = prof[i]
            res[k] = d
        return res

    # ---- individually exposed steps (device tensors) ---------------------------------------
    def lcl(self, p, t, td, options=None):
        opts = options if options is not None else make_options()
        p, t, td = [x.contiguous() for x in torch.broadcast_tensors(p, t, td)]
        out = torch.empty((3,) + tuple(p.shape), dtype=p.dtype, device=p.device)
        st = self.lib.xp_lcl(self.handle, p.data_ptr(), t.data_ptr(), td.data_ptr(), p.numel(),
                             _dtype_code(p), ctypes.byref(opts), out[0].data_ptr(), out[1].data_ptr(),
                             out[2].data_ptr(), self._stream())
        self._check(st, "xp_lcl")
        return out[0], out[1], out[2]

    def moist_lapse(self, pressure, parcel_temperature, parcel_pressure):
        pressure = pressure.contiguous()
        L, N = pressure.shape
        pt = parcel_temperature.expand(N).contiguous()
        pp = parcel_pressure.expand(N).contiguous()
        out = torch.empty_like(pressure)
        st = self.lib.xp_moist_lapse(self.handle, pressure.data_ptr(), N, L, N, _dtype_code(pressure),
                                     pt.data_ptr(), pp.data_ptr(), out.data_ptr(), N, self._stream())
        self._check(st, "xp_moist_lapse")
        return out

    def parcel_profile(self, pressure, parcel_pressure, parcel_temperature, parcel_dewpoint,
                       options=None):
        opts = options if options is not None else make_options()
        pressure = pressure.contiguous()
        L, N = pressure.shape
        pp = parcel_pressure.expand(N).contiguous()
        pt = parcel_temperature.expand(N).contiguous()
        pd = parcel_dewpoint.expand(N).contiguous()
        out = torch.empty((2, L, N), dtype=pressure.dtype, device=pressure.device)
        lcl = torch.empty((3, N), dtype=pressure.dtype, device=pressure.device)
        pin = XpParcelIn(pp.data_ptr(), pt.data_ptr(), pd.data_ptr())
        st = self.lib.xp_parcel_profile(self.handle, pressure.data_ptr(), N, L, N, _dtype_code(pressure),
                                        ctypes.byref(pin), ctypes.byref(opts), out[0].data_ptr(),
                                        out[1].data_ptr(), N, lcl[0].data_ptr(), lcl[1].data_ptr(),
                                        lcl[2].data_ptr(), self._stream())
        self._check(st, "xp_parcel_profile")
        return {"temperature": out[0], "virtual_temperature": out[1], "lcl_pressure": lcl[0],
                "lcl_temperature": lcl[1], "lcl_virtual_temperature": lcl[2]}

    def lfc_el(self, pressure, parcel_temperature, temperature, lcl_pressure, lcl_temperature):
        pressure, parcel_temperature, temperature = [x.contiguous() for x in
                                                     (pressure, parcel_temperature, temperature)]
        L, N = pressure.shape
        lp = lcl_pressure.expand(N).contiguous()
        lt = lcl_temperature.expand(N).contiguous()
        out = torch.empty((4, N), dtype=pressure.dtype, device=pressure.device)
        st = self.lib.xp_lfc_el(self.handle, pressure.data_ptr(), parcel_temperature.data_ptr(),
                                temperature.data_ptr(), N, L, N, _dtype_code(pressure), lp.data_ptr(),
                                lt.data_ptr(), out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(),
                                out[3].data_ptr(), self._stream())
        self._check(st, "xp_lfc_el")
        return {"lfc_pressure": out[0], "lfc_temperature": out[1], "el_pressure": out[2],
                "el_temperature": out[3]}

    def cape_cin_base(self, pressure, temperature, lfc_pressure, el_pressure, parcel_temperature,
                      options=None):
        opts = options if options is not None else make_options()
        pressure, temperature, parcel_temperature = [x.contiguous() for x in
                                                     (pressure, temperature, parcel_temperature)]
        L, N = pressure.shape
        lf = lfc_pressure.expand(N).contiguous()
        el = el_pressure.expand(N).contiguous()
        out = torch.empty((2, N), dtype=pressure.dtype, device=pressure.device)
        st = self.lib.xp_cape_cin_base(self.handle, pressure.data_ptr(), temperature.data_ptr(),
                                       parcel_temperature.data_ptr(), N, L, N, _dtype_code(pressure),
                                       lf.data_ptr(), el.data_ptr(), ctypes.byref(opts),
                                       out[0].data_ptr(), out[1].data_ptr(), self._stream())
        self._check(st, "xp_cape_cin_base")
        return {"cape": out[0], "cin": out[1]}


    # ---- derived-index helpers (device tensors) -----------------------------------------------------
    def interp_levels(self, coords, fields, at, log=False):
        """linear_interp / log_interp (PF:1758-1828) of up to 4 fields [L, N] at one coordinate value per
        column.  ``coords``: [L, N] or shared [L]; ``at``: float or [N] tensor.  Returns a list of [N]."""
        fields = [x.contiguous() for x in fields]
        L, N = fields[0].shape
        dt = fields[0].dtype
        assert 1 <= len(fields) <= 4 and all(x.shape == (L, N) and x.dtype == dt for x in fields)
        coords = coords.to(dt).contiguous()
        c1d = coords.dim() == 1
        outs = [torch.empty((N,), dtype=dt, device=fields[0].device) for _ in fields]
        fp = (c_void_p * len(fields))(*[x.data_ptr() for x in fields])
        op = (c_void_p * len(fields))(*[x.data_ptr() for x in outs])
        if isinstance(at, torch.Tensor):
            at_t = at.to(dt).expand(N).contiguous()
            at_ptr, at_s = at_t.data_ptr(), 0.0
        else:
            at_t, at_ptr, at_s = None, None, float(at)
        st = self.lib.xp_interp_levels(self.handle, coords.data_ptr(), 1 if c1d else N, int(c1d), fp, op,
                                       len(fields), N, L, N, _dtype_code(fields[0]), at_ptr, at_s, int(bool(log)),
                                       self._stream())
        self._check(st, "xp_interp_levels")
        return outs

    def level_crossing(self, coords, field, level):
        """Lowest coordinate at which ``field`` [L, N] crosses ``level`` (PF:992-1064 + min, PF:2153)."""
        field = field.contiguous()
        L, N = field.shape
        coords = coords.to(field.dtype).contiguous()
        c1d = coords.dim() == 1
        out = torch.empty((N,), dtype=field.dtype, device=field.device)
        st = self.lib.xp_level_crossing(self.handle, coords.data_ptr(), 1 if c1d else N, int(c1d),
                                        field.data_ptr(), N, L, N, _dtype_code(field), float(level),
                                        out.data_ptr(), self._stream())
        self._check(st, "xp_level_crossing")
        return out

    # ---- layer primitives (xp_layers.cu) ---------------------------------------------------------------
    def mixed_layer(self, pressure, fields, depth=100.0, pressure_field=-1):
        """mixed_layer (PF:137-162) of up to 4 variables [L, N] per call (more: several calls).  ``pressure``:
        [L, N] or shared [L]; ``pressure_field``: index of the variable that is the pressure itself, or -1.
        Returns a list of [N] tensors."""
        fields = [x.contiguous() for x in fields]
        L, N = fields[0].shape
        dt = fields[0].dtype
        assert all(x.shape == (L, N) and x.dtype == dt for x in fields)
        pressure = pressure.to(dt).contiguous()
        p1d = pressure.dim() == 1
        outs = []
        for g in range(0, len(fields), 4):
            grp = fields[g:g + 4]
            o = [torch.empty((N,), dtype=dt, device=grp[0].device) for _ in grp]
            fp = (c_void_p * len(grp))(*[x.data_ptr() for x in grp])
            op = (c_void_p * len(grp))(*[x.data_ptr() for x in o])
            st = self.lib.xp_mixed_layer(self.handle, pressure.data_ptr(), 1 if p1d else N, int(p1d), fp, op,
                                         len(grp), pressure_field - g if g <= pressure_field < g + 4 else -1, N, L, N,
                                         _dtype_code(grp[0]), float(depth), self._stream())
            self._check(st, "xp_mixed_layer")
            outs += o
        return outs

    def mixed_parcel(self, pressure, temperature, dewpoint, depth=100.0):
        """mixed_parcel (PF:229-289): dict of the six [N] variables the reference returns."""
        temperature = temperature.contiguous()
        L, N = temperature.shape
        dt = temperature.dtype
        dewpoint = dewpoint.to(dt).contiguous()
        pressure = pressure.to(dt).contiguous()
        p1d = pressure.dim() == 1
        outs = {n: torch.empty((N,), dtype=dt, device=temperature.device) for n in MIXED_PARCEL_FIELDS}
        o = XpMixedParcelOut(*[outs[n].data_ptr() for n in MIXED_PARCEL_FIELDS])
        st = self.lib.xp_mixed_parcel(self.handle, pressure.data_ptr(), 1 if p1d else N, int(p1d),
                                      temperature.data_ptr(), dewpoint.data_ptr(), N, L, N, _dtype_code(temperature),
                                      float(depth), ctypes.byref(o), self._stream())
        self._check(st, "xp_mixed_parcel")
        return outs

    def layer_bounds(self, pressure, n_columns, depth=100.0, interpolate=True):
        """(bottom, top) pressures of get_layer (PF:63-100; bound_pressure PF:208-227 when not interpolating)."""
        pressure = pressure.contiguous()
        p1d = pressure.dim() == 1
        L = pressure.shape[0]
        N = int(n_columns)
        bottom = torch.empty((N,), dtype=pressure.dtype, device=pressure.device)
        top = torch.empty_like(bottom)
        st = self.lib.xp_layer_bounds(self.handle, pressure.data_ptr(), 1 if p1d else N, int(p1d), L, N,
                                      _dtype_code(pressure), float(depth), int(bool(interpolate)),
                                      bottom.data_ptr(), top.data_ptr(), self._stream())
        self._check(st, "xp_layer_bounds")
        return bottom, top

    def downdraft_cape(self, pressure, temperature, dewpoint, metpy_compat="1.4.1", profile=False, outputs=None):
        """Downdraft CAPE (xp_downdraft_cape) of the columns of ``temperature`` / ``dewpoint`` [L, N] on ``pressure``
        ([L, N] or a shared [L]; any level stride).  Returns a dict of the DOWNDRAFT_FIELDS [N] and, with
        ``profile``, 'downdraft_parcel_temperature' [L, N].  ``outputs`` (a subset of those names) leaves the others
        uncomputed (NULL in the call)."""
        compat = {"1.4.1": 141, "1.6.2": 162, 141: 141, 162: 162, "141": 141, "162": 162}[metpy_compat]
        L, N = temperature.shape
        dt = temperature.dtype
        dewpoint = dewpoint.to(dt)
        if not (temperature.stride(1) == 1 and dewpoint.stride(1) == 1 and temperature.stride(0) == dewpoint.stride(0)):
            temperature, dewpoint = temperature.contiguous(), dewpoint.contiguous()
        pressure = pressure.to(dt)
        p1d = pressure.dim() == 1
        if not p1d and pressure.stride(1) != 1:
            pressure = pressure.contiguous()
        names = list(DOWNDRAFT_FIELDS) + (["downdraft_parcel_temperature"] if profile else [])
        if outputs is not None:
            names = [n for n in names if n in outputs]
        dev = temperature.device
        res = {n: torch.empty((L, N) if n == "downdraft_parcel_temperature" else (N,), dtype=dt, device=dev)
               for n in names}
        ptr = {n: res[n].data_ptr() if n in res else None
               for n in DOWNDRAFT_FIELDS + ["downdraft_parcel_temperature"]}
        o = XpDowndraftOut(ptr["dcape"], ptr["downdraft_start_pressure"], ptr["downdraft_start_temperature"],
                           ptr["downdraft_parcel_temperature"], N)
        st = self.lib.xp_downdraft_cape(self.handle, pressure.data_ptr(), pressure.stride(0), int(p1d),
                                        temperature.data_ptr(), dewpoint.data_ptr(), temperature.stride(0), L, N,
                                        _dtype_code(temperature), compat, ctypes.byref(o), self._stream())
        self._check(st, "xp_downdraft_cape")
        return res

    def effective_inflow_layer(self, p, t, td, options=None, min_cape=100.0, min_cin=-250.0, profile=False,
                               outputs=None):
        """Effective inflow layer (xp_effective_inflow_layer) of the device columns ``t`` / ``td`` [L, N] on ``p``
        ([L, N] or a shared [L]).  Returns a dict of the EFFECTIVE_FIELDS [N] (base and top pressure) and, with
        ``profile``, the EFFECTIVE_LEVEL_FIELDS [L, N] (CAPE / CIN of the parcel of every level; this lifts every
        valid level of every column).  ``outputs`` (a subset of those names) leaves the others uncomputed (NULL in the
        call).  ``options``: make_options(...) (most_unstable_depth selects the gate's parcel)."""
        opts = options if options is not None else make_options()
        cols, L, N = self._columns(p, t, td)
        names = list(EFFECTIVE_FIELDS) + (list(EFFECTIVE_LEVEL_FIELDS) if profile else [])
        if outputs is not None:
            names = [n for n in names if n in outputs]
        res = {n: torch.empty((L, N) if n in EFFECTIVE_LEVEL_FIELDS else (N,), dtype=t.dtype, device=t.device)
               for n in names}
        ptr = {n: res[n].data_ptr() if n in res else None for n in EFFECTIVE_FIELDS + EFFECTIVE_LEVEL_FIELDS}
        o = XpEffectiveOut(ptr["effective_inflow_base"], ptr["effective_inflow_top"], ptr["level_parcel_cape"],
                           ptr["level_parcel_cin"], N)
        st = self.lib.xp_effective_inflow_layer(self.handle, ctypes.byref(cols), ctypes.byref(opts), float(min_cape),
                                                float(min_cin), ctypes.byref(o), self._stream())
        self._check(st, "xp_effective_inflow_layer")
        return res
    # ---- level primitives (xp_levels.cu) ---------------------------------------------------------------
    @staticmethod
    def _ptrs(tensors):
        return (c_void_p * max(len(tensors), 1))(*[x.data_ptr() for x in tensors])

    def insert_level(self, coords, level_coord, fields, level_values):
        """insert_level (PF:933-990): ``coords`` [L, N] or [L]; ``level_coord`` [N]; ``fields`` list of [L, N] with
        their values ``level_values`` (list of [N]) at the new level.  Returns (coords_out, [outputs]) with L + 1
        levels."""
        dt, dev = level_coord.dtype, level_coord.device
        N = level_coord.shape[0]
        coords = coords.to(dt).contiguous()
        L = coords.shape[0]
        c1d = coords.dim() == 1
        fields = [x.to(dt).contiguous() for x in fields]
        level_values = [x.to(dt).contiguous() for x in level_values]
        assert len(fields) == len(level_values) and all(x.shape == (L, N) for x in fields)
        cout = torch.empty((L + 1, N), dtype=dt, device=dev)
        outs = [torch.empty((L + 1, N), dtype=dt, device=dev) for _ in fields]
        for g in range(0, max(len(fields), 1), 4):
            grp, lv, o = fields[g:g + 4], level_values[g:g + 4], outs[g:g + 4]
            st = self.lib.xp_insert_level(self.handle, coords.data_ptr(), 1 if c1d else N, int(c1d),
                                          level_coord.contiguous().data_ptr(), self._ptrs(grp), self._ptrs(lv),
                                          self._ptrs(o), len(grp), cout.data_ptr() if g == 0 else None, N, N, L, N,
                                          _dtype_code(level_coord), self._stream())
            self._check(st, "xp_insert_level")
        return cout, outs

    def shift_out_nans(self, ref, fields):
        """shift_out_nans (PF:1699-1720).  Returns ([shifted fields], level_shift int32 [N])."""
        ref = ref.contiguous()
        L, N = ref.shape
        fields = [x.to(ref.dtype).contiguous() for x in fields]
        outs = [torch.empty_like(x) for x in fields]
        shift = torch.empty((N,), dtype=torch.int32, device=ref.device)
        for g in range(0, max(len(fields), 1), 4):
            grp, o = fields[g:g + 4], outs[g:g + 4]
            st = self.lib.xp_shift_out_nans(self.handle, ref.data_ptr(), self._ptrs(grp), self._ptrs(o), len(grp), N,
                                            L, N, _dtype_code(ref), shift.data_ptr(), self._stream())
            self._check(st, "xp_shift_out_nans")
        return outs, shift

    def trapz(self, x, fields, mask=None, sign=0):
        """trapz (PF:164-206) of the [L, N] ``fields`` along ``x`` ([L, N] or shared [L]); ``mask``: bool/uint8
        [>= L-1, N] labelled by the lower level.  Returns a list of [N]."""
        fields = [v.contiguous() for v in fields]
        L, N = fields[0].shape
        dt = fields[0].dtype
        x = x.to(dt).contiguous()
        x1d = x.dim() == 1
        if mask is not None:
            mask = mask.to(torch.uint8).contiguous()
            assert mask.shape[0] >= L - 1 and mask.shape[1] == N
        outs = [torch.empty((N,), dtype=dt, device=v.device) for v in fields]
        for g in range(0, len(fields), 4):
            grp, o = fields[g:g + 4], outs[g:g + 4]
            st = self.lib.xp_trapz(self.handle, x.data_ptr(), 1 if x1d else N, int(x1d), self._ptrs(grp),
                                   self._ptrs(o), len(grp), N, L, N, _dtype_code(grp[0]),
                                   mask.data_ptr() if mask is not None else None, N, int(sign), self._stream())
            self._check(st, "xp_trapz")
        return outs

    def find_intersections(self, x, a, b, log_x=False):
        """find_intersections (PF:992-1064): dict of the six [L-1, N] arrays (row r = interval r..r+1)."""
        a = a.contiguous()
        L, N = a.shape
        b = b.to(a.dtype).expand(L, N).contiguous()
        x = x.to(a.dtype).contiguous()
        x1d = x.dim() == 1
        outs = {n: torch.full((max(L - 1, 0), N), float("nan"), dtype=a.dtype, device=a.device)
                for n in INTERSECTION_FIELDS}
        o = XpIntersectionsOut(*[outs[n].data_ptr() for n in INTERSECTION_FIELDS])
        st = self.lib.xp_find_intersections(self.handle, x.data_ptr(), 1 if x1d else N, int(x1d), a.data_ptr(),
                                            b.data_ptr(), N, N, L, N, _dtype_code(a), int(bool(log_x)),
                                            ctypes.byref(o), self._stream())
        self._check(st, "xp_find_intersections")
        return outs

    def interp1d(self, at, xp, fp):
        """interp1d_numba (PF:23-37): numpy.interp along the last axis of ``at`` [..., m] with ``xp`` ([n] or
        [..., n], increasing) and ``fp`` [..., n]."""
        dt = fp.dtype
        lead = torch.broadcast_shapes(at.shape[:-1], fp.shape[:-1])
        m, n = at.shape[-1], fp.shape[-1]
        at2 = at.to(dt).expand(*lead, m).reshape(-1, m).contiguous()
        fp2 = fp.expand(*lead, n).reshape(-1, n).contiguous()
        x1d = xp.dim() == 1
        xp2 = xp.to(dt).contiguous() if x1d else xp.to(dt).expand(*lead, n).reshape(-1, n).contiguous()
        out = torch.empty_like(at2)
        st = self.lib.xp_interp1d(self.handle, at2.data_ptr(), xp2.data_ptr(), int(x1d), fp2.data_ptr(), out.data_ptr(),
                                  at2.shape[0], m, n, _dtype_code(fp2), self._stream())
        self._check(st, "xp_interp1d")
        return out.reshape(*lead, m)

    def trap_around_zeros(self, x, y, log_x=True):
        """trap_around_zeros (PF:1200-1289): (dict of the five [2L-1, N] area arrays, bool mask [L, N])."""
        y = y.contiguous()
        L, N = y.shape
        x = x.to(y.dtype).contiguous()
        x1d = x.dim() == 1
        outs = {n: torch.empty((2 * L - 1, N), dtype=y.dtype, device=y.device) for n in ZERO_AREA_FIELDS}
        mask = torch.empty((L, N), dtype=torch.uint8, device=y.device)
        o = XpZeroAreasOut(*([outs[n].data_ptr() for n in ZERO_AREA_FIELDS] + [mask.data_ptr()]))
        st = self.lib.xp_trap_around_zeros(self.handle, x.data_ptr(), 1 if x1d else N, int(x1d), y.data_ptr(), N, N, L,
                                           N, _dtype_code(y), int(bool(log_x)), ctypes.byref(o), self._stream())
        self._check(st, "xp_trap_around_zeros")
        return outs, mask != 0

    def valid_data(self, pressure, n_columns):
        """The pressure check of valid_data (PF:2320); the verdict arrives through take_flags()."""
        pressure = pressure.contiguous()
        p1d = pressure.dim() == 1
        st = self.lib.xp_valid_data(self.handle, pressure.data_ptr(), 1 if p1d else int(n_columns), int(p1d),
                                    pressure.shape[0], int(n_columns), _dtype_code(pressure), self._stream())
        self._check(st, "xp_valid_data")

    # ---- pointwise helpers (device tensors of one shape and dtype) -------------------------------------
    def _pointwise(self, fn_name, inputs, extra=()):
        """Call lib.<fn_name>(ctx, *inputs, n, dtype, *extra, out, stream) on broadcast, contiguous inputs."""
        dt = inputs[0].dtype
        xs = [x.to(dt) for x in inputs]
        xs = [x.contiguous() for x in torch.broadcast_tensors(*xs)]
        out = torch.empty_like(xs[0])
        st = getattr(self.lib, fn_name)(self.handle, *[x.data_ptr() for x in xs], xs[0].numel(), _dtype_code(xs[0]),
                                        *extra, out.data_ptr(), self._stream())
        self._check(st, fn_name)
        return out

    def dewpoint_from_specific_humidity(self, pressure, temperature, specific_humidity, metpy_compat="1.4.1"):
        compat = {"1.4.1": 141, "1.6.2": 162, 141: 141, 162: 162, "141": 141, "162": 162}[metpy_compat]
        # dtype follows the temperature
        pressure = pressure.to(temperature.dtype)
        return self._pointwise("xp_dewpoint_from_specific_humidity", [pressure, temperature, specific_humidity],
                               (compat,))

    def saturation_mixing_ratio(self, pressure, temperature):
        return self._pointwise("xp_saturation_mixing_ratio", [pressure, temperature])

    def dry_lapse(self, pressure, parcel_temperature, parcel_pressure):
        return self._pointwise("xp_dry_lapse", [pressure, parcel_temperature, parcel_pressure])

    def mixing_ratio(self, temperature, dewpoint, pressure, metpy_compat="1.4.1"):
        compat = {"1.4.1": 141, "1.6.2": 162, 141: 141, 162: 162, "141": 141, "162": 162}[metpy_compat]
        return self._pointwise("xp_mixing_ratio", [temperature, dewpoint, pressure], (compat,))

    def virtual_temperature(self, temperature, mixing_ratio, epsilon=0.608):
        dt = temperature.dtype
        t, w = [x.contiguous() for x in torch.broadcast_tensors(temperature, mixing_ratio.to(dt))]
        out = torch.empty_like(t)
        st = self.lib.xp_virtual_temperature(self.handle, t.data_ptr(), w.data_ptr(), t.numel(), _dtype_code(t),
                                             float(epsilon), out.data_ptr(), self._stream())
        self._check(st, "xp_virtual_temperature")
        return out

    def wet_bulb_temperature(self, pressure, temperature, dewpoint):
        return self._pointwise("xp_wet_bulb_temperature", [pressure, temperature, dewpoint])

    def significant_hail_parameter(self, mucape, mixing_ratio, lapse, temp_500, shear, flh):
        return self._pointwise("xp_significant_hail_parameter", [mucape, mixing_ratio, lapse, temp_500, shear, flh])

    def storm_proxies(self, fields):
        """``fields``: dict of the PROXY_INPUTS tensors (one shape).  Returns dict of 9 bool tensors + 'ship'."""
        dt = fields["mixed_100_cape"].dtype
        xs = [fields[k].to(dt) for k in PROXY_INPUTS]
        xs = [x.contiguous() for x in torch.broadcast_tensors(*xs)]
        n = xs[0].numel()
        flags = [torch.empty(xs[0].shape, dtype=torch.uint8, device=xs[0].device) for _ in PROXY_FLAGS]
        ship = torch.empty_like(xs[0])
        inp = XpProxyInputs(*[x.data_ptr() for x in xs])
        outp = XpProxyOutputs(*([f.data_ptr() for f in flags] + [ship.data_ptr()]))
        st = self.lib.xp_storm_proxies(self.handle, ctypes.byref(inp), n, _dtype_code(xs[0]), ctypes.byref(outp),
                                       self._stream())
        self._check(st, "xp_storm_proxies")
        res = {k: f.bool() for k, f in zip(PROXY_FLAGS, flags)}
        res["ship"] = ship
        return res


_contexts = {}
_ctx_lock = threading.Lock()


def get_context(device=None):
    """Process-wide context per device (the reference keeps its tables in module globals, PF:18-21)."""
    if device is None:
        device = torch.cuda.current_device() if torch.cuda.is_available() else 0
    device = int(device)
    with _ctx_lock:
        if device not in _contexts:
            _contexts[device] = Context(device)
        return _contexts[device]
