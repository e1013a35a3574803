"""Drop-in host layer for the parcel path of ``modules/parcel_functions.py`` ("PF").

Same function names, argument meaning, defaults, returned variable names/attrs and
``AssertionError`` messages as the reference, for the hot path named in BASELINE.json.  The
work is done by hand-written sm_100a kernels behind the C ABI of ``libxparcel.so``
(include/xparcel.h); this module only unwraps arrays into level-major buffers and wraps
the results.  There is no CPU implementation here: without the CUDA library or a GPU every
compute call raises.

Accepted inputs
  * ``xarray.DataArray`` (when xarray is installed): ``vert_dim`` names the vertical
    dimension; results are ``xarray.Dataset``/``DataArray`` with the same dims/coords.
  * ``numpy.ndarray`` / ``torch.Tensor``: ``vert_axis`` (default 0) is the vertical axis;
    results come back in a ``Dataset`` (a dict with attribute access) of the same array
    type.  CUDA tensors are used in place (zero copy); host arrays go through the
    library's pinned staging pipeline.

Units: hPa and K (README.md:9).  Level 0 is the surface; pressure must decrease with level.
"""

import numpy as np
import torch

from . import _lib

try:  # optional: the reference's container types
    import xarray as _xr
except Exception:  # pragma: no cover - xarray is absent in the build image
    _xr = None

__all__ = ["load_moist_adiabat_lookups", "lookup_tables_loaded", "moist_adiabat_tables", "lcl",
           "dry_lapse", "moist_lapse", "mixing_ratio", "virtual_temperature", "parcel_profile",
           "parcel_profile_with_lcl", "lfc_el", "cape_cin_base", "cape_cin",
           "surface_based_cape_cin", "mixed_layer_cape_cin", "most_unstable_cape_cin",
           "mixed_parcel", "most_unstable_parcel", "mix_layer", "from_most_unstable_parcel",
           "parcel_suite", "parcel_suite_chunks", "Dataset", "linear_interp", "log_interp", "lifted_index",
           "deep_convective_index", "isobar_temperature", "lapse_rate", "freezing_level_height",
           "melting_level_height", "wet_bulb_temperature_fast", "wind_shear",
           "dewpoint_from_specific_humidity", "conv_properties", "min_conv_properties", "downdraft_cape",
           "effective_inflow_layer", "bunkers_storm_motion", "storm_relative_helicity", "effective_layer_parameters",
           "supercell_composite_parameter", "significant_tornado_parameter"]

KAPPA = 0.28571428571428564       # metpy.constants.kappa (PF:313)

# variable metadata of the reference (PF:669-677, 769-770, 849-852, 1188-1196, 1366-1385)
_ATTRS = {
    "lcl_pressure": {"long_name": "Lifting condensation level pressure", "units": "hPa"},
    "lcl_temperature": {"long_name": "Lifting condensation level temperature", "units": "K"},
    "lcl_virtual_temperature": {"long_name": "Lifting condensation level virtual temperature",
                                "units": "K"},
    "lfc_pressure": {"long_name": "Level of free convection pressure", "units": "hPa"},
    "lfc_temperature": {"long_name": "Level of free convection temperature", "units": "K"},
    "el_pressure": {"long_name": "Equilibrium level pressure", "units": "hPa"},
    "el_temperature": {"long_name": "Equilibrium level temperature", "units": "K"},
    "cape": {"long_name": "Convective available potential energy", "units": "J kg$^{-1}$"},
    "cin": {"long_name": "Convective inhibition", "units": "J kg$^{-1}$"},
    "pressure": {"long_name": "Pressure at LCL"},                       # PF:890 (sic)
    "temperature": {"long_name": "Temperature at LCL", "units": "K"},   # PF:889 (sic)
    "virtual_temperature": {"long_name": "Virtual temperature", "units": "K"},
    "environment_temperature": {"long_name": "Environment temperature", "units": "K"},
    "environment_dewpoint": {"long_name": "Environment dewpoint", "units": "K"},
    "environment_virtual_temperature": {"long_name": "Virtual temperature", "units": "K"},
    "dcape": {"long_name": "Downdraft convective available potential energy", "units": "J kg$^{-1}$"},
    "downdraft_start_pressure": {"long_name": "Downdraft source pressure", "units": "hPa"},
    "downdraft_start_temperature": {"long_name": "Downdraft source wet-bulb temperature", "units": "K"},
    "downdraft_parcel_temperature": {"long_name": "Downdraft parcel temperature", "units": "K"},
    "effective_inflow_base": {"long_name": "Effective inflow layer base pressure", "units": "hPa"},
    "effective_inflow_top": {"long_name": "Effective inflow layer top pressure", "units": "hPa"},
    "level_parcel_cape": {"long_name": "CAPE of the parcel lifted from each level", "units": "J kg$^{-1}$"},
    "level_parcel_cin": {"long_name": "CIN of the parcel lifted from each level", "units": "J kg$^{-1}$"},
    "bunkers_right_u": {"long_name": "Bunkers right-mover storm motion, eastward", "units": "m s$^{-1}$"},
    "bunkers_right_v": {"long_name": "Bunkers right-mover storm motion, northward", "units": "m s$^{-1}$"},
    "bunkers_left_u": {"long_name": "Bunkers left-mover storm motion, eastward", "units": "m s$^{-1}$"},
    "bunkers_left_v": {"long_name": "Bunkers left-mover storm motion, northward", "units": "m s$^{-1}$"},
    "mean_wind_u": {"long_name": "0-6 km mean wind, eastward", "units": "m s$^{-1}$"},
    "mean_wind_v": {"long_name": "0-6 km mean wind, northward", "units": "m s$^{-1}$"},
    "effective_srh": {"long_name": "Effective storm-relative helicity", "units": "m$^{2}$ s$^{-2}$"},
    "effective_bulk_wind_difference": {"long_name": "Effective bulk wind difference", "units": "m s$^{-1}$"},
    "supercell_composite_parameter": {"long_name": "Supercell composite parameter", "units": "1"},
    "significant_tornado_parameter": {"long_name": "Significant tornado parameter (effective layer, with CIN)",
                                      "units": "1"},
}


class Dataset(dict):
    """Minimal stand-in for ``xarray.Dataset`` when inputs are plain arrays: a dict of arrays
    with attribute access, ``attrs`` and per-variable ``var_attrs``."""

    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.attrs = {}
        self.var_attrs = {}

    def __getattr__(self, name):
        try:
            return self[name]
        except KeyError as e:
            raise AttributeError(name) from e

    def rename(self, mapping):
        out = Dataset((mapping.get(k, k), v) for k, v in self.items())
        out.attrs = dict(self.attrs)
        out.var_attrs = {mapping.get(k, k): v for k, v in self.var_attrs.items()}
        return out


# ----------------------------------------------------------------------------- table state
def load_moist_adiabat_lookups(device=None, tables=None, **kwargs):
    """PF:39-54.  Build the two moist-adiabat lookup tables on the GPU (PF:447-523 takes ~100 s
    of SciPy solves; the CUDA builder a few ms), or install caller-provided ones
    (``tables=(index_grid uint16 [2196, 7150], curves float32 [14300, 2196])``)."""
    ctx = _lib.get_context(device)
    if tables is not None:
        ctx.tables_set(tables[0], tables[1])
    else:
        ctx.tables_build()
    return ctx


def lookup_tables_loaded(device=None):
    """PF:56-61."""
    assert _lib.get_context(device).tables_loaded(), "Call load_moist_adiabat_lookups first."


def moist_adiabat_tables(regenerate=False, cache=True, device=None, **kwargs):
    """PF:318-356: returns (index_grid, curves) as NumPy arrays (uint16 [2196, 7150] on descending
    pressure x temperature, float32 [14300, 2196] on ascending pressure)."""
    ctx = _lib.get_context(device)
    if regenerate or not ctx.tables_loaded():
        ctx.tables_build()
    return ctx.tables_get()


def moist_adiabat_lookup(pressure_levels=None, temperatures=None, pres_step=0.5, temp_step=0.02, device=None):
    """PF:447-523 on the reference's default grids (pressures 1100 ... 2.5 hPa in 0.5 hPa steps, temperatures 173 ...
    315.98 K in 0.02 K steps -- the only ones the CUDA builder and the kernels' table addressing support): builds the
    tables on the GPU and returns (index_grid, curves) like ``moist_adiabat_tables``."""
    if pressure_levels is not None:
        ref = np.round(np.arange(1100, 2, step=-0.5), 1)
        assert np.shape(pressure_levels) == ref.shape and np.allclose(pressure_levels, ref), \
            "only the reference's default pressure_levels are supported"
    if temperatures is not None:
        ref = np.round(np.arange(173, 316, step=0.02), 2)
        assert np.shape(temperatures) == ref.shape and np.allclose(temperatures, ref), \
            "only the reference's default temperatures are supported"
    assert pres_step == 0.5 and temp_step == 0.02, "only the reference's default steps are supported"
    ctx = _lib.get_context(device)
    ctx.tables_build()
    return ctx.tables_get()


def round_to(x, to, dp=2):
    """PF:358-362: round ``x`` to the nearest ``to``, then to ``dp`` decimals (host helper of the table grid)."""
    return np.round(np.round(np.asarray(x) / to) * to, dp)


# ----------------------------------------------------------------------------- (un)wrapping
class _Layout:
    """How an input field maps to level-major [L, N] blocks and how results map back."""

    def __init__(self, template, vert_dim, vert_axis):
        self.is_xr = _xr is not None and isinstance(template, _xr.DataArray)
        self.template = template
        if self.is_xr:
            self.vert_dim = vert_dim
            self.vert_axis = template.dims.index(vert_dim) if vert_dim in template.dims else None
            arr = template.data
        else:
            self.vert_dim = vert_dim
            self.vert_axis = vert_axis
            arr = template
        self.is_torch = isinstance(arr, torch.Tensor)
        self.shape = tuple(arr.shape)
        va = self.vert_axis
        self.L = self.shape[va] if va is not None else 1
        self.col_shape = tuple(s for i, s in enumerate(self.shape) if i != va)

    def to_block(self, x, device, dtype):
        """Any input -> torch tensor [L, N] (or [L] for a 1-D pressure axis), level-major."""
        if self.is_xr and _xr is not None and isinstance(x, _xr.DataArray):
            if x.dims != self.template.dims:
                if set(x.dims) == {self.vert_dim}:
                    x = x.data
                    t = torch.as_tensor(np.asarray(x)) if not isinstance(x, torch.Tensor) else x
                    return t.to(dtype)
                x = x.broadcast_like(self.template).transpose(*self.template.dims)
            x = x.data
        if not isinstance(x, torch.Tensor):
            x = np.asarray(x)
            if x.dtype not in (np.float32, np.float64):
                x = x.astype(np.float64)
            x = torch.from_numpy(np.ascontiguousarray(x)) if x.ndim else torch.tensor(float(x))
        if x.dtype != dtype:
            x = x.to(dtype)
        if x.dim() == 1 and len(self.shape) > 1 and x.shape[0] == self.L:
            return x                                          # shared 1-D vertical axis
        if tuple(x.shape) != self.shape:
            x = x.expand(self.shape)
        va = self.vert_axis
        if va != 0:
            x = x.movedim(va, 0)
        x = x.reshape(self.L, -1)
        if x.shape[1] > 1 and x.stride(1) != 1:
            x = x.contiguous()
        if x.shape[0] > 1 and x.stride(0) < x.shape[1]:
            x = x.contiguous()
        return x

    def scalar_to_block(self, x, dtype):
        """Per-column quantity (no vertical dim) -> torch [N]."""
        if self.is_xr and _xr is not None and isinstance(x, _xr.DataArray):
            dims = tuple(d for d in self.template.dims if d != self.vert_dim)
            if x.dims != dims:
                x = x.broadcast_like(self.template.isel({self.vert_dim: 0}, drop=True)).transpose(*dims)
            x = x.data
        if not isinstance(x, torch.Tensor):
            x = torch.as_tensor(np.asarray(x, dtype=np.float64))
        x = x.to(dtype)
        n = int(np.prod(self.col_shape)) if self.col_shape else 1
        if x.numel() == 1:
            return x.reshape(1).expand(n)
        return x.expand(self.col_shape).reshape(n)

    def _finish(self, t):
        if self.is_torch:
            return t
        return t.cpu().numpy() if t.is_cuda else t.numpy()

    def wrap_scalar(self, t, name):
        t = self._finish(t.reshape(self.col_shape))
        if self.is_xr:
            dims = tuple(d for d in self.template.dims if d != self.vert_dim)
            coords = {k: v for k, v in self.template.coords.items()
                      if self.vert_dim not in v.dims}
            return _xr.DataArray(t, dims=dims, coords=coords, name=name, attrs=dict(_ATTRS.get(name, {})))
        return t

    def wrap_profile(self, t, name, n_levels):
        """[n_levels, N] -> original dim order with the vertical axis re-labelled 0..n-1
        offset by the template's first label (PF:968-970)."""
        va = self.vert_axis if self.vert_axis is not None else 0
        t = t[:n_levels].reshape((n_levels,) + self.col_shape)
        if va != 0:
            t = t.movedim(0, va)
        t = self._finish(t)
        if self.is_xr:
            first = self.template[self.vert_dim].values[0] if self.vert_dim in self.template.coords else 0
            coords = {k: v for k, v in self.template.coords.items() if self.vert_dim not in v.dims}
            coords[self.vert_dim] = np.arange(n_levels) + first
            return _xr.DataArray(t, dims=self.template.dims, coords=coords, name=name,
                                 attrs=dict(_ATTRS.get(name, {})))
        return t

    def dataset(self, variables):
        if self.is_xr:
            return _xr.Dataset(variables)
        ds = Dataset(variables)
        ds.var_attrs = {k: dict(_ATTRS.get(k, {})) for k in variables}
        return ds


def _prepare(pressure, temperature, dewpoint, vert_dim, vert_axis, device):
    lay = _Layout(temperature, vert_dim, vert_axis)
    raw = temperature.data if lay.is_xr else temperature
    if isinstance(raw, torch.Tensor):
        dtype = raw.dtype if raw.dtype in (torch.float32, torch.float64) else torch.float64
        dev = raw.device
    else:
        raw = np.asarray(raw)
        dtype = torch.float32 if raw.dtype == np.float32 else torch.float64
        dev = torch.device("cpu")
    t = lay.to_block(temperature, dev, dtype)
    td = lay.to_block(dewpoint, dev, dtype)
    p = lay.to_block(pressure, dev, dtype)
    if t.stride(0) != td.stride(0):
        td = td.contiguous()
        t = t.contiguous()
    ctx = _lib.get_context(device if device is not None else (dev.index if dev.type == "cuda" else None))
    return lay, ctx, p.to(dev), t, td


def _options(kwargs):
    known = ("virtual_temperature_correction", "lcl_interp", "pos_cape_neg_cin", "post_zero_cin",
             "metpy_compat")
    return {k: kwargs[k] for k in known if k in kwargs}


def _clear_flags(ctx):
    """The reference-assert flags live in one word per context that only take_flags() clears: drop whatever an
    earlier call that never collected them (direct Context use, another function) left behind, so that every
    function of this module reports its OWN launches only."""
    ctx.take_flags()


def _check_flags(ctx):
    flags = ctx.take_flags()
    assert not (flags & _lib.FLAG_PRESSURES_NOT_UNIQUE), "Vertical pressures are not unique"   # PF:131
    assert not (flags & _lib.FLAG_TOP_TEMPERATURE_NAN), "Top temperature is NaN."              # PF:1149


_PROFILE_VARS = [("pressure", "profile_pressure"), ("temperature", "profile_temperature"),
                 ("virtual_temperature", "profile_virtual_temperature"),
                 ("environment_temperature", "profile_environment_temperature"),
                 ("environment_virtual_temperature", "profile_environment_virtual_temperature"),
                 ("environment_dewpoint", "profile_environment_dewpoint")]
_SCALAR_VARS = ["lcl_pressure", "lcl_temperature", "lcl_virtual_temperature", "lfc_pressure",
                "lfc_temperature", "el_pressure", "el_temperature"]


def _profile_levels(kind, res, L):
    """Vertical length of the returned profile: the reference trims levels that are NaN in
    every column with dropna(how='all') before lifting (PF:1552, PF:1637)."""
    if kind in ("sb", "explicit"):
        return L + 1
    shift = res["level_shift"]
    min_shift = int(shift.min().item()) if shift.numel() else 0
    min_shift = min(min_shift, L - 1) if kind == "mu" else min(min_shift, L)
    return (L - min_shift) + (1 if kind == "ml" else 0) + 1


def _run(kind, pressure, temperature, dewpoint, vert_dim, vert_axis, device, profile, explicit=None,
         depth=None, specific_humidity=False, **kwargs):
    lay, ctx, p, t, td = _prepare(pressure, temperature, dewpoint, vert_dim, vert_axis, device)
    _clear_flags(ctx)
    okw = _options(kwargs)
    if depth is not None:
        okw["mixed_layer_depth" if kind == "ml" else "most_unstable_depth"] = depth
    opts = _lib.make_options(**okw)
    ex = None
    if explicit is not None:
        ex = [lay.scalar_to_block(e, t.dtype).to(t.device) for e in explicit]
    res = ctx.cape_cin(p, t, td, kinds=(kind,), options=opts, profile=profile, explicit=ex,
                       specific_humidity=specific_humidity)[kind]
    _check_flags(ctx)
    cc = lay.dataset({"cape": lay.wrap_scalar(res["cape"], "cape"),
                      "cin": lay.wrap_scalar(res["cin"], "cin")})
    vtc = okw.get("virtual_temperature_correction", True)
    cc.attrs["correction"] = ("Virtual temperature correction used in CAPE/CIN calculations." if vtc else
                              "Virtual temperature correction not used in CAPE/CIN calculations.")
    pv = {}
    if profile:
        n_lev = _profile_levels(kind, res, lay.L)
        for name, key in _PROFILE_VARS:
            pv[name] = lay.wrap_profile(res[key], name, n_lev)
    for name in _SCALAR_VARS:
        pv[name] = lay.wrap_scalar(res[name], name)
    prof = lay.dataset(pv)
    parcel = lay.dataset({"pressure": lay.wrap_scalar(res["parcel_pressure"], "pressure"),
                          "temperature": lay.wrap_scalar(res["parcel_temperature"], "temperature"),
                          "dewpoint": lay.wrap_scalar(res["parcel_dewpoint"], "dewpoint")})
    return cc, prof, parcel, lay, res


def _describe(cc, cape_desc, cin_desc, prefix):
    if isinstance(cc, Dataset):
        cc.var_attrs.setdefault("cape", {})["description"] = cape_desc
        cc.var_attrs.setdefault("cin", {})["description"] = cin_desc
    else:
        cc["cape"].attrs["description"] = cape_desc
        cc["cin"].attrs["description"] = cin_desc
    if prefix is not None:
        cc = cc.rename({"cape": prefix + "_cape", "cin": prefix + "_cin"})
    return cc


# ----------------------------------------------------------------------------- public API
def cape_cin(pressure, temperature, dewpoint, parcel_temperature, parcel_pressure, parcel_dewpoint,
             vert_dim="model_level_number", virtual_temperature_correction=True, lcl_interp="log",
             vert_axis=0, device=None, profile=True, **kwargs):
    """PF:1394-1475.  Returns (Dataset{cape, cin}, profile Dataset incl. LCL/LFC/EL)."""
    cc, prof, _, _, _ = _run("explicit", pressure, temperature, dewpoint, vert_dim, vert_axis, device,
                             profile, explicit=(parcel_pressure, parcel_temperature, parcel_dewpoint),
                             virtual_temperature_correction=virtual_temperature_correction,
                             lcl_interp=lcl_interp, **kwargs)
    return cc, prof


def surface_based_cape_cin(pressure, temperature, dewpoint, vert_dim="model_level_number", prefix=None,
                           vert_axis=0, device=None, profile=True, **kwargs):
    """PF:1477-1514."""
    cc, prof, _, _, _ = _run("sb", pressure, temperature, dewpoint, vert_dim, vert_axis, device,
                             profile, **kwargs)
    cc = _describe(cc, "CAPE for surface-based parcel.", "CIN for surface-based parcel.", prefix)
    return cc, prof


def mixed_layer_cape_cin(pressure, temperature, dewpoint, vert_dim="model_level_number", depth=100,
                         prefix=None, vert_axis=0, device=None, profile=True, **kwargs):
    """PF:1651-1697.  Returns (cape_cin, profile, mixed parcel)."""
    cc, prof, mp, _, _ = _run("ml", pressure, temperature, dewpoint, vert_dim, vert_axis, device,
                              profile, depth=depth, **kwargs)
    desc = f"fully-mixed lowest {depth} hPa parcel"
    cc = _describe(cc, f"CAPE for {desc}.", f"CIN for {desc}", prefix)
    return cc, prof, mp


def most_unstable_cape_cin(pressure, temperature, dewpoint, vert_dim="model_level_number", depth=300,
                           prefix=None, vert_axis=0, device=None, profile=True, **kwargs):
    """PF:1557-1602.  Returns (cape_cin, profile, unstable_layer)."""
    cc, prof, ul, _, _ = _run("mu", pressure, temperature, dewpoint, vert_dim, vert_axis, device,
                              profile, depth=depth, **kwargs)
    desc = f"most-unstable parcel in lowest {depth} hPa."
    cc = _describe(cc, f"CAPE for {desc}", f"CIN for {desc}", prefix)
    return cc, prof, ul


def parcel_profile_with_lcl(pressure, temperature, dewpoint, parcel_pressure, parcel_temperature,
                            parcel_dewpoint, vert_dim="model_level_number", lcl_interp="log",
                            vert_axis=0, device=None, **kwargs):
    """PF:806-856."""
    _, prof, _, _, _ = _run("explicit", pressure, temperature, dewpoint, vert_dim, vert_axis, device,
                            True, explicit=(parcel_pressure, parcel_temperature, parcel_dewpoint),
                            lcl_interp=lcl_interp, **kwargs)
    for k in ("lfc_pressure", "lfc_temperature", "el_pressure", "el_temperature"):
        if isinstance(prof, Dataset):
            prof.pop(k, None)
        else:
            prof = prof.drop_vars(k)
    return prof


def mixed_parcel(pressure, temperature, dewpoint, depth=100, vert_dim="model_level_number",
                 vert_axis=0, device=None, **kwargs):
    """PF:229-289: Dataset{theta, mixing_ratio, temperature, vapour_pressure, dewpoint, pressure} of the fully
    mixed lowest ``depth`` hPa (``xp_mixed_parcel``; pressure = the level-0 pressure, PF:287)."""
    lay, ctx, p, t, td = _prepare(pressure, temperature, dewpoint, vert_dim, vert_axis, device)
    on_gpu = t.is_cuda
    res = ctx.mixed_parcel(p.cuda(), t.cuda(), td.cuda(), depth=depth)
    return lay.dataset({k: lay.wrap_scalar(v if on_gpu else v.cpu(), k) for k, v in res.items()})


def mixed_layer(dat, depth=100, vert_dim="model_level_number", vert_axis=0, device=None):
    """PF:137-162: mass-weighted mean over the lowest ``depth`` hPa of every variable of ``dat`` (a Dataset or
    dict that contains 'pressure'; like the reference's, the result also holds the mean of 'pressure' itself)."""
    names = _names(dat)
    assert "pressure" in names, "dat must contain pressure."
    template = next((dat[k] for k in names if getattr(dat[k], "ndim", 0) > 1), dat["pressure"])
    ctx = _lib.get_context(device)
    lay, dtype, on_gpu = _layout_of(template, vert_dim, vert_axis)
    blocks = _blocks(lay, [dat[k] for k in names], dtype)
    pb = blocks[names.index("pressure")]
    n = int(np.prod(lay.col_shape)) if lay.col_shape else 1
    full = [b if b.dim() == 2 else b[:, None].expand(lay.L, n).contiguous() for b in blocks]
    res = ctx.mixed_layer(pb, full, depth=depth, pressure_field=names.index("pressure"))
    return lay.dataset({k: lay.wrap_scalar(v if on_gpu else v.cpu(), k) for k, v in zip(names, res)})


def _names(dat):
    return list(dat.data_vars) if hasattr(dat, "data_vars") else list(dat.keys())


def _template(arrays):
    """The array whose shape is the columns' shape: the first of ``arrays`` with more than one dimension, so that a
    shared 1-D pressure axis next to [L, N] fields lays out as the fields do (else the first array)."""
    return next((a for a in arrays if getattr(a, "ndim", 0) > 1), arrays[0])


def _full_blocks(lay, blocks):
    n = int(np.prod(lay.col_shape)) if lay.col_shape else 1
    return [b if b.dim() == 2 else b[:, None].expand(lay.L, n).contiguous() for b in blocks]


def insert_level(d, level, coords, vert_dim="model_level_number", fill_value=-999, vert_axis=0, device=None):
    """PF:933-990: insert ``level`` (values of ``coords`` and of the variables to keep, one per column) into the
    vertically sorted ``d``; the result holds the keys of ``level`` on L + 1 levels."""
    assert fill_value == -999, "only the reference's default fill_value is implemented"
    keys = _names(level)
    ctx = _lib.get_context(device)
    others = [k for k in keys if k != coords]
    lay, dtype, on_gpu = _layout_of(_template([d[coords]] + [d[k] for k in others]), vert_dim, vert_axis)
    blocks = _full_blocks(lay, _blocks(lay, [d[coords]] + [d[k] for k in others], dtype))
    lev = [lay.scalar_to_block(level[k], dtype).cuda().contiguous() for k in [coords] + others]
    assert not bool((blocks[0] == fill_value).any()), "dataset d contains fill_value."          # PF:962
    cout, outs = ctx.insert_level(blocks[0], lev[0], blocks[1:], lev[1:])
    res = dict(zip([coords] + others, [cout] + outs))
    return lay.dataset({k: lay.wrap_profile(res[k] if on_gpu else res[k].cpu(), k, lay.L + 1) for k in keys})


def add_lcl_to_profile(profile, vert_dim="model_level_number", environment=None, interpolator="log", vert_axis=0,
                       device=None, metpy_compat="1.4.1"):
    """PF:858-931: insert the LCL level into a ``parcel_profile`` result (pressure, temperature,
    virtual_temperature + lcl_*) and, if given, into the ``environment`` (interpolated at the LCL pressure, its
    virtual temperature recomputed from the interpolated temperature and dewpoint, PF:911-920).  The fused kernel
    behind ``parcel_profile_with_lcl`` does all of this in one pass; this is the step on its own, composed of
    ``xp_insert_level``, ``xp_interp_levels``, ``xp_mixing_ratio`` and ``xp_virtual_temperature``."""
    assert interpolator in ["linear", "log"], "interpolator must be linear or log"
    ctx = _lib.get_context(device)
    lay, dtype, on_gpu = _layout_of(profile["pressure"], vert_dim, vert_axis)
    pv = ["pressure", "temperature", "virtual_temperature"]
    pb, tb, tvb = _full_blocks(lay, _blocks(lay, [profile[k] for k in pv], dtype))
    lcl = [lay.scalar_to_block(profile["lcl_" + k], dtype).cuda().contiguous() for k in pv]
    assert not bool((pb == -999).any()), "dataset d contains fill_value."                       # PF:962
    cout, (tout, tvout) = ctx.insert_level(pb, lcl[0], [tb, tvb], lcl[1:])                      # PF:884
    fin = lambda v: v if on_gpu else v.cpu()
    out = {k: lay.wrap_profile(fin(v), k, lay.L + 1) for k, v in zip(pv, (cout, tout, tvout))}
    for k, v in zip(pv, lcl):
        out["lcl_" + k] = lay.wrap_scalar(fin(v), "lcl_" + k)
    if environment is not None:
        names = [k for k in _names(environment) if k != "pressure"]
        blocks = _full_blocks(lay, _blocks(lay, [environment["pressure"]] + [environment[k] for k in names], dtype))
        eb, fields = blocks[0], blocks[1:]
        lev = []
        for g in range(0, len(fields), 4):
            lev += ctx.interp_levels(eb, fields[g:g + 4], lcl[0], log=(interpolator == "log"))  # PF:899-906
        if "virtual_temperature" in names:                                                      # PF:911-920
            mr = ctx.mixing_ratio(lev[names.index("temperature")], lev[names.index("dewpoint")], lcl[0],
                                  metpy_compat=metpy_compat)
            lev[names.index("virtual_temperature")] = ctx.virtual_temperature(lev[names.index("temperature")], mr)
        assert not bool((eb == -999).any()), "dataset d contains fill_value."
        _, eouts = ctx.insert_level(eb, lcl[0], fields, lev)                                    # PF:923
        for k, v in zip(names, eouts):
            out["environment_" + k] = lay.wrap_profile(fin(v), "environment_" + k, lay.L + 1)
    return lay.dataset(out)


def shift_out_nans(x, name, dim="model_level_number", vert_axis=0, device=None):
    """PF:1699-1720: shift every variable of ``x`` down, column by column, until level 0 of ``name`` is not NaN."""
    names = _names(x)
    ctx = _lib.get_context(device)
    lay, dtype, on_gpu = _layout_of(_template([x[name]] + [x[k] for k in names]), dim, vert_axis)
    blocks = _full_blocks(lay, _blocks(lay, [x[k] for k in names], dtype))
    outs, _ = ctx.shift_out_nans(blocks[names.index(name)], blocks)
    return lay.dataset({k: lay.wrap_profile(o if on_gpu else o.cpu(), k, lay.L) for k, o in zip(names, outs)})


def trapz(dat, x, dim="model_level_number", mask=None, only_positive=False, only_negative=False, vert_axis=0,
          device=None):
    """PF:164-206: trapezoidal integral of every variable of ``dat`` along its variable ``x``; ``mask`` selects the
    intervals (labelled by their lower level)."""
    assert not (only_positive and only_negative), "Only negative OR positive regions can be included in trapz."
    names = _names(dat)
    ctx = _lib.get_context(device)
    template = next((dat[k] for k in names if getattr(dat[k], "ndim", 0) > 1), dat[x])
    lay, dtype, on_gpu = _layout_of(template, dim, vert_axis)
    blocks = _blocks(lay, [dat[k] for k in names], dtype)
    xb = blocks[names.index(x)]
    mb = None
    if mask is not None:
        m = mask.data if (_xr is not None and isinstance(mask, _xr.DataArray)) else mask
        m = m if isinstance(m, torch.Tensor) else torch.as_tensor(np.asarray(m))
        va = lay.vert_axis or 0
        mb = m.movedim(va, 0).reshape(m.shape[va], -1).cuda() != 0
    res = ctx.trapz(xb, _full_blocks(lay, blocks), mask=mb, sign=1 if only_positive else (-1 if only_negative else 0))
    return lay.dataset({k: lay.wrap_scalar(v if on_gpu else v.cpu(), k) for k, v in zip(names, res)})


def find_intersections(x, a, b, dim="model_level_number", log_x=False, vert_axis=0, device=None):
    """PF:992-1064: crossings of the curves ``a`` and ``b`` over ``x``.  Returns a Dataset of all_intersect_x/y,
    increasing_x/y and decreasing_x/y on L - 1 levels labelled, like the reference's offset_dim, by the upper level
    of each interval."""
    ctx = _lib.get_context(device)
    lay, dtype, on_gpu = _layout_of(a, dim, vert_axis)
    xb, ab, bb = _blocks(lay, [x, a, b], dtype)
    (ab, bb) = _full_blocks(lay, [ab, bb])
    res = ctx.find_intersections(xb, ab, bb, log_x=log_x)
    out = {}
    for k, v in res.items():
        w = lay.wrap_profile(v if on_gpu else v.cpu(), k, lay.L - 1)
        if lay.is_xr:
            w = w.assign_coords({dim: w[dim] + 1})                                     # PF:1026 offset labels
        out[k] = w
    return lay.dataset(out)


def trap_around_zeros(x, y, dim="model_level_number", log_x=True, start=0, vert_axis=0, device=None):
    """PF:1200-1289 (``start`` = 0): the half-areas next to every zero of ``y`` along ``x``.  Returns (areas, mask):
    areas holds area, x, dx, x_from, x_to on 2L - 1 levels (the before-zero parts labelled by the lower level, then
    the after-zero parts), mask [L] is True where the ordinary trapezoid above a level stays in the integral."""
    assert start == 0, "only start=0 (the reference's own use) is implemented"
    ctx = _lib.get_context(device)
    lay, dtype, on_gpu = _layout_of(y, dim, vert_axis)
    xb, yb = _blocks(lay, [x, y], dtype)
    (yb,) = _full_blocks(lay, [yb])
    res, mask = ctx.trap_around_zeros(xb, yb, log_x=log_x)
    fin = lambda v: v if on_gpu else v.cpu()
    areas = lay.dataset({k: lay.wrap_profile(fin(v), k, 2 * lay.L - 1) for k, v in res.items()})
    return areas, lay.wrap_profile(fin(mask), "mask", lay.L)


def interp1d_numba(at, xp, fp, device=None):
    """PF:23-37: ``numpy.interp(at, xp, fp)`` along the last axis, broadcasting over the leading ones like the
    reference's gufunc ``(m),(n),(n)->(m)`` (here a CUDA kernel, ``xp_interp1d``)."""
    ctx = _lib.get_context(device)
    on_gpu = isinstance(fp, torch.Tensor) and fp.is_cuda
    is_t = isinstance(fp, torch.Tensor)
    dt = _float_dtype([fp])
    conv = lambda a: (a if isinstance(a, torch.Tensor) else torch.as_tensor(np.asarray(a))).to(dt).cuda()  # noqa: E731
    out = ctx.interp1d(conv(at), conv(xp), conv(fp))
    return out if on_gpu else (out.cpu() if is_t else out.cpu().numpy())


def valid_data(dat, vert_dim="model_level_number", vert_axis=0, device=None):
    """PF:2308-2321: True if the vertical index steps by one and the pressures decrease with the level number."""
    if hasattr(dat, "coords") and vert_dim in getattr(dat, "coords", {}):
        assert np.all(np.abs(np.diff(np.asarray(dat[vert_dim]))) == 1), "Index increments must all be 1."
    ctx = _lib.get_context(device)
    lay, dtype, _ = _layout_of(dat["pressure"], vert_dim, vert_axis)
    (pb,) = _blocks(lay, [dat["pressure"]], dtype)
    n = int(np.prod(lay.col_shape)) if lay.col_shape else 1
    _clear_flags(ctx)
    ctx.valid_data(pb, n)
    flags = ctx.take_flags()
    assert (flags & _lib.FLAG_PRESSURE_ORDER_CHECKED) and not (flags & _lib.FLAG_PRESSURE_NOT_DECREASING), \
        "Pressures must decrease with increasing level number."
    return True


def get_layer(dat, depth=100, vert_dim="model_level_number", interpolate=True, vert_axis=0, device=None):
    """PF:63-100: the lowest ``depth`` hPa of ``dat`` (which must contain 'pressure'), everything else NaN.  With
    ``interpolate`` the layer top is interpolated in ln p and inserted (L + 1 levels), otherwise the top is the
    level closest to it (bound_pressure)."""
    names = _names(dat)
    ctx = _lib.get_context(device)
    lay, dtype, on_gpu = _layout_of(_template([dat["pressure"]] + [dat[k] for k in names]), vert_dim, vert_axis)
    blocks = _full_blocks(lay, _blocks(lay, [dat[k] for k in names], dtype))
    pb = blocks[names.index("pressure")]
    n = pb.shape[1]
    bottom, top = ctx.layer_bounds(pb, n, depth=depth, interpolate=interpolate)
    n_lev = lay.L
    if interpolate:
        others = [k for k in names if k != "pressure"]
        ob = [blocks[names.index(k)] for k in others]
        lev = []
        for g in range(0, len(ob), 4):
            lev += ctx.interp_levels(pb, ob[g:g + 4], top, log=True)                 # PF:85
        cout, outs = ctx.insert_level(pb, top, ob, lev)                               # PF:87-90
        res = dict(zip(["pressure"] + others, [cout] + outs))
        blocks = [res[k] for k in names]
        pb = cout
        n_lev += 1
    keep = (pb <= bottom[None, :]) & (pb >= top[None, :])                             # PF:97-98
    nanv = torch.full((), float("nan"), dtype=pb.dtype, device=pb.device)
    out = {k: torch.where(keep, b, nanv) for k, b in zip(names, blocks)}
    return lay.dataset({k: lay.wrap_profile(v if on_gpu else v.cpu(), k, n_lev) for k, v in out.items()})


def bound_pressure(pressure, bound=None, vert_dim="model_level_number", vert_axis=0, device=None, depth=None):
    """PF:208-227 as get_layer(interpolate=False) uses it (PF:92-94): the level pressure closest to
    ``bottom - depth``, the larger one on a tie.  Pass ``depth``; an arbitrary ``bound`` array is not supported."""
    assert bound is None and depth is not None, "only bound = bottom pressure - depth (pass depth=) is implemented"
    ctx = _lib.get_context(device)
    lay, dtype, on_gpu = _layout_of(pressure, vert_dim, vert_axis)
    (pb,) = _blocks(lay, [pressure], dtype)
    n = int(np.prod(lay.col_shape)) if lay.col_shape else 1
    _, top = ctx.layer_bounds(pb, n, depth=depth, interpolate=False)
    return lay.wrap_scalar(top if on_gpu else top.cpu(), "pressure")


def most_unstable_parcel(dat=None, depth=300, vert_dim="model_level_number", pressure=None,
                         temperature=None, dewpoint=None, vert_axis=0, device=None, **kwargs):
    """PF:102-135.  ``dat`` is a Dataset/dict with pressure, temperature and dewpoint."""
    if dat is not None:
        pressure, temperature, dewpoint = dat["pressure"], dat["temperature"], dat["dewpoint"]
    _, _, ul, _, _ = _run("mu", pressure, temperature, dewpoint, vert_dim, vert_axis, device, False,
                          depth=depth, **kwargs)
    return ul


def _lifted_columns(kind, pressure, temperature, dewpoint, vert_dim, depth, vert_axis, device, **kwargs):
    """The lifted column of mix_layer (PF:1604-1649) / from_most_unstable_parcel (PF:1517-1555) is
    the environment part of the profile without its LCL level; the host removes that level."""
    cc, prof, parcel, lay, res = _run(kind, pressure, temperature, dewpoint, vert_dim, vert_axis, device,
                                      True, depth=depth, **kwargs)
    L = lay.L
    n_lev = _profile_levels(kind, res, L)
    P = res["profile_pressure"][:n_lev]
    lcl_p = res["lcl_pressure"]
    # index of the inserted LCL level: number of levels with p >= lcl_p (PF:965)
    pos = ((P >= lcl_p[None, :]).sum(dim=0) - 1).clamp(min=0)
    # the inserted level is the LAST level with p >= lcl among equal pressures
    n = n_lev - 1
    idx = torch.arange(n, device=P.device)[:, None]
    src = idx + (idx >= pos[None, :]).to(idx.dtype)
    bad = torch.isnan(lcl_p)
    src = torch.where(bad[None, :], idx.expand(-1, P.shape[1]), src)
    out = {}
    for name, key in (("pressure", "profile_pressure"), ("temperature", "profile_environment_temperature"),
                      ("dewpoint", "profile_environment_dewpoint")):
        out[name] = lay.wrap_profile(torch.gather(res[key][:n_lev], 0, src), name, n)
    return out["pressure"], out["temperature"], out["dewpoint"], parcel


def mix_layer(pressure, temperature, dewpoint, vert_dim="model_level_number", depth=100, load=True,
              vert_axis=0, device=None, **kwargs):
    """PF:1604-1649: (pressure, temperature, dewpoint) with the mixed parcel as the bottom level and
    the mixed layer removed, plus the mixed parcel.  Columns whose parcel is NaN come back as NaN."""
    return _lifted_columns("ml", pressure, temperature, dewpoint, vert_dim, depth, vert_axis, device,
                           **kwargs)


def from_most_unstable_parcel(pressure, temperature, dewpoint, vert_dim="model_level_number", depth=300,
                              vert_axis=0, device=None, **kwargs):
    """PF:1517-1555."""
    return _lifted_columns("mu", pressure, temperature, dewpoint, vert_dim, depth, vert_axis, device,
                           **kwargs)


def parcel_suite(pressure, temperature, dewpoint, vert_dim="model_level_number", vert_axis=0,
                 device=None, mixed_layer_depth=100, most_unstable_depth=300, specific_humidity=False, **kwargs):
    """Surface-based + mixed-layer + most-unstable CAPE/CIN/LCL/LFC/EL in ONE pass over the columns
    (the hot-path part of parcel_test.py:416-547 ``conv_properties_xarray``; no profile output).
    Returns a Dataset with the reference's prefixed names: surface_*, mixed_100_*, max_*.
    ``specific_humidity=True``: ``dewpoint`` holds specific humidity [kg/kg] -- model output (p, T, q) is consumed
    directly, converted in the kernels' load stage (parcel_test.py:432-436 computes the dewpoint first)."""
    lay, ctx, p, t, td = _prepare(pressure, temperature, dewpoint, vert_dim, vert_axis, device)
    opts = _lib.make_options(mixed_layer_depth=mixed_layer_depth, most_unstable_depth=most_unstable_depth,
                             **_options(kwargs))
    _clear_flags(ctx)
    res = ctx.cape_cin(p, t, td, kinds=("sb", "ml", "mu"), options=opts, profile=False,
                       specific_humidity=specific_humidity)
    _check_flags(ctx)
    out = {}
    prefixes = {"sb": "surface", "ml": f"mixed_{int(mixed_layer_depth)}", "mu": "max"}
    for kind, pre in prefixes.items():
        for name in ["cape", "cin"] + _SCALAR_VARS:
            out[f"{pre}_{name}"] = lay.wrap_scalar(res[kind][name], name)
        if kind != "sb":
            for name in ("pressure", "temperature", "dewpoint"):
                out[f"{pre}_parcel_{name}"] = lay.wrap_scalar(res[kind]["parcel_" + name], name)
    return lay.dataset(out)


def parcel_suite_chunks(blocks, mixed_layer_depth=100, most_unstable_depth=300, workers=2, device=None,
                        specific_humidity=False, **kwargs):
    """``parcel_suite`` over a CHUNKED source: ``blocks`` is an iterable of (pressure, temperature, dewpoint) column
    blocks, level-major [L, n_i] -- NumPy / memmap / zarr / dask arrays or anything with ``.compute()`` /
    ``__array__`` (``streaming.iter_column_blocks`` cuts big lazy arrays into such blocks without reading them).
    Yields one ``Dataset`` of host arrays per block, in order, with the names of ``parcel_suite``.  Blocks are read,
    uploaded, lifted and downloaded concurrently (xarray_parcel_b200/streaming.py) -- the stand-in for the
    reference's dask ``map_blocks`` execution (PF:585-592, 667)."""
    from . import streaming
    opts = _lib.make_options(mixed_layer_depth=mixed_layer_depth, most_unstable_depth=most_unstable_depth,
                             **_options(kwargs))
    prefixes = {"sb": "surface", "ml": f"mixed_{int(mixed_layer_depth)}", "mu": "max"}
    for res in streaming.suite_blocks(blocks, kinds=("sb", "ml", "mu"), workers=workers, device=device,
                                      options=opts, specific_humidity=specific_humidity):
        out = Dataset()
        for kind, pre in prefixes.items():
            for name in ["cape", "cin"] + _SCALAR_VARS:
                out[f"{pre}_{name}"] = res[kind][name].numpy()
            if kind != "sb":
                for name in ("pressure", "temperature", "dewpoint"):
                    out[f"{pre}_parcel_{name}"] = res[kind]["parcel_" + name].numpy()
        out.var_attrs = {k: dict(_ATTRS.get(k.split("_", 1)[-1], {})) for k in out}
        yield out


# ---- individually exposed steps ---------------------------------------------------------------
def _to_dev(x, like=None, dtype=None):
    if _xr is not None and isinstance(x, _xr.DataArray):
        x = x.data
    if not isinstance(x, torch.Tensor):
        x = torch.as_tensor(np.asarray(x, dtype=np.float64 if dtype is None else None))
    if dtype is not None:
        x = x.to(dtype)
    elif x.dtype not in (torch.float32, torch.float64):
        x = x.to(torch.float64)
    if not x.is_cuda:
        x = x.cuda()
    return x


def _back(t, template):
    raw = template.data if (_xr is not None and isinstance(template, _xr.DataArray)) else template
    if isinstance(raw, torch.Tensor):
        return t if raw.is_cuda else t.cpu()
    return t.cpu().numpy()


def _float_dtype(args):
    """The dtype of a step's computation: that of the first float32 / float64 tensor or float32 NumPy array among
    ``args`` (NumPy float64, Python scalars and other types compute in float64)."""
    for a in args:
        a = a.data if (_xr is not None and isinstance(a, _xr.DataArray)) else a
        if isinstance(a, torch.Tensor) and a.dtype in (torch.float32, torch.float64):
            return a.dtype
        if isinstance(a, np.ndarray) and a.dtype == np.float32:
            return torch.float32
    return torch.float64


def _pointwise(method, args, template=0, name=None, attrs=None, device=None, **kw):
    """Run a pointwise Context method (``_lib.Context.<method>``: one CUDA thread per point) on broadcast
    inputs and hand the result back as the template's array type (DataArray / torch / NumPy)."""
    ctx = _lib.get_context(device)
    tmpl = args[template]
    if _xr is not None and any(isinstance(a, _xr.DataArray) for a in args):
        xa = _xr.broadcast(*[a if isinstance(a, _xr.DataArray) else _xr.DataArray(a) for a in args])
        tmpl = xa[template]
        args = [a.data for a in xa]
    dt = _float_dtype(args)
    dev = [_to_dev(a, dtype=dt) for a in args]
    res = getattr(ctx, method)(*dev, **kw)
    if _xr is not None and isinstance(tmpl, _xr.DataArray):
        out = tmpl.copy(data=res.cpu().numpy())
        out.attrs = dict(attrs or {})
        if name:
            out.name = name
        return out
    raw = args[template]
    if isinstance(raw, torch.Tensor):
        return res if raw.is_cuda else res.cpu()
    return res.cpu().numpy()


def lcl(parcel_pressure, parcel_temperature, parcel_dewpoint, device=None, **kwargs):
    """PF:609-682.  Returns Dataset{lcl_pressure, lcl_temperature, lcl_virtual_temperature}."""
    ctx = _lib.get_context(device)
    dt = _float_dtype([parcel_temperature, parcel_pressure, parcel_dewpoint])
    pt, pp, pd = [_to_dev(x, dtype=dt) for x in (parcel_temperature, parcel_pressure, parcel_dewpoint)]
    a, b, c = ctx.lcl(pp, pt, pd, _lib.make_options(**_options(kwargs)))
    ds = Dataset({"lcl_pressure": _back(a, parcel_temperature), "lcl_temperature": _back(b, parcel_temperature),
                  "lcl_virtual_temperature": _back(c, parcel_temperature)})
    ds.var_attrs = {k: dict(_ATTRS[k]) for k in ds}
    return ds


def dry_lapse(pressure, parcel_temperature, parcel_pressure=None, vert_dim="model_level_number",
              vert_axis=0, device=None):
    """PF:291-316: T0 * (p / p0) ** kappa (``xp_dry_lapse``, one thread per point)."""
    if parcel_pressure is None:
        if _xr is not None and isinstance(pressure, _xr.DataArray):
            parcel_pressure = pressure.max(vert_dim)
        elif isinstance(pressure, torch.Tensor):
            parcel_pressure = pressure.amax(dim=vert_axis, keepdim=True)
        else:
            parcel_pressure = np.max(pressure, axis=vert_axis, keepdims=True)
    return _pointwise("dry_lapse", [pressure, parcel_temperature, parcel_pressure], name="temperature",
                      attrs={"long_name": "Dry lapse rate temperature", "units": "K"}, device=device)


def virtual_temperature(temperature, mixing_ratio, epsilon=0.608, device=None):
    """PF:782-804 (``xp_virtual_temperature``)."""
    return _pointwise("virtual_temperature", [temperature, mixing_ratio], name="virtual_temperature",
                      attrs={"long_name": "Virtual temperature", "units": "K"}, device=device, epsilon=epsilon)


def mixing_ratio(temperature, dewpoint, pressure, metpy_compat="1.4.1", device=None):
    """PF:684-710: relative humidity from the dewpoint, then mixing ratio from relative humidity
    (``xp_mixing_ratio``; MetPy 1.4.1 or >= 1.6 form of mixing_ratio_from_relative_humidity)."""
    return _pointwise("mixing_ratio", [temperature, dewpoint, pressure], name="mixing_ratio",
                      attrs={"long_name": "Mixing ratio", "units": "kg kg$^{-1}$"}, device=device,
                      metpy_compat=metpy_compat)


def _lift_layout(pressure, parcels, vert_dim, vert_axis):
    """Layout of a lift of ``parcels`` over ``pressure``.  A shared 1-D pressure axis under parcels of more than one
    element takes its columns from the parcels: the profiles come back with the vertical dimension first, then the
    parcels' dimensions, as if the axis had been broadcast against them."""
    lay = _Layout(pressure, vert_dim, vert_axis)
    if len(lay.shape) != 1:
        return lay
    raw_of = lambda x: x.data if (_xr is not None and isinstance(x, _xr.DataArray)) else x     # noqa: E731
    shape_of = lambda x: tuple(x.shape) if isinstance(x, torch.Tensor) else np.shape(x)      # noqa: E731
    par = next((x for x in parcels if x is not None and int(np.prod(shape_of(raw_of(x)))) > 1), None)
    if par is None:
        return lay
    if lay.is_xr and isinstance(par, _xr.DataArray):
        tmpl = _xr.broadcast(pressure, par)[0]
        tmpl = tmpl.transpose(vert_dim, *[d for d in tmpl.dims if d != vert_dim])
        return _Layout(tmpl, vert_dim, 0)
    shape = shape_of(raw_of(par))
    raw = pressure.data if lay.is_xr else pressure
    lead = (slice(None),) + (None,) * len(shape)
    if isinstance(raw, torch.Tensor):
        tmpl = raw[lead].expand(raw.shape[0], *shape)
    else:
        raw = np.asarray(raw)
        tmpl = np.broadcast_to(raw[lead], raw.shape + shape)
    return _Layout(tmpl, vert_dim, 0)


def _lift_pressure(lay, pressure, dtype):
    """Pressure of a lift as a contiguous CUDA block [L, N] (a shared axis broadcast over the layout's columns)."""
    p = lay.to_block(pressure, None, dtype).cuda()
    if p.dim() == 1:
        n = int(np.prod(lay.col_shape)) if lay.col_shape else 1
        p = p[:, None].expand(p.shape[0], n)
    return p.contiguous()


def moist_lapse(pressure, parcel_temperature, parcel_pressure=None, vert_dim="model_level_number",
                persist=True, vert_axis=0, device=None):
    """PF:525-607: lookup-table moist adiabat.  ``pressure`` is [L, ...] (vertical axis first for
    plain arrays)."""
    ctx = _lib.get_context(device)
    lookup_tables_loaded(device)
    lay = _lift_layout(pressure, (parcel_temperature, parcel_pressure), vert_dim, vert_axis)
    raw = pressure.data if lay.is_xr else pressure
    dtype = raw.dtype if isinstance(raw, torch.Tensor) else (torch.float32 if np.asarray(raw).dtype == np.float32 else torch.float64)
    p = _lift_pressure(lay, pressure, dtype)
    if parcel_pressure is None:
        parcel_pressure = p[0]
        pp = parcel_pressure
    else:
        pp = lay.scalar_to_block(parcel_pressure, dtype).cuda()
    pt = lay.scalar_to_block(parcel_temperature, dtype).cuda()
    out = ctx.moist_lapse(p.contiguous(), pt, pp)
    return lay.wrap_profile(out if isinstance(raw, torch.Tensor) and raw.is_cuda else out.cpu(),
                            "temperature", lay.L)


def parcel_profile(pressure, parcel_pressure, parcel_temperature, parcel_dewpoint,
                   vert_dim="model_level_number", vert_axis=0, device=None, **kwargs):
    """PF:712-780: parcel temperature / virtual temperature on the input levels + the LCL."""
    ctx = _lib.get_context(device)
    lookup_tables_loaded(device)
    lay = _lift_layout(pressure, (parcel_pressure, parcel_temperature, parcel_dewpoint), vert_dim, vert_axis)
    raw = pressure.data if lay.is_xr else pressure
    dtype = raw.dtype if isinstance(raw, torch.Tensor) else (torch.float32 if np.asarray(raw).dtype == np.float32 else torch.float64)
    on_gpu = isinstance(raw, torch.Tensor) and raw.is_cuda
    p = _lift_pressure(lay, pressure, dtype)
    pp = lay.scalar_to_block(parcel_pressure, dtype).cuda()
    pt = lay.scalar_to_block(parcel_temperature, dtype).cuda()
    pd = lay.scalar_to_block(parcel_dewpoint, dtype).cuda()
    r = ctx.parcel_profile(p.contiguous(), pp, pt, pd, _lib.make_options(**_options(kwargs)))
    fix = (lambda x: x) if on_gpu else (lambda x: x.cpu())
    out = {"pressure": lay.wrap_profile(fix(p.contiguous()), "pressure", lay.L),
           "temperature": lay.wrap_profile(fix(r["temperature"]), "temperature", lay.L),
           "virtual_temperature": lay.wrap_profile(fix(r["virtual_temperature"]), "virtual_temperature", lay.L)}
    for k in ("lcl_pressure", "lcl_temperature", "lcl_virtual_temperature"):
        out[k] = lay.wrap_scalar(fix(r[k]), k)
    return lay.dataset(out)


def lfc_el(pressure, parcel_temperature, temperature, lcl_pressure, lcl_temperature,
           vert_dim="model_level_number", vert_axis=0, device=None):
    """PF:1066-1198 on caller-supplied parcel and environment temperature profiles."""
    ctx = _lib.get_context(device)
    lay = _Layout(temperature, vert_dim, vert_axis)
    raw = temperature.data if lay.is_xr else temperature
    dtype = raw.dtype if isinstance(raw, torch.Tensor) else (torch.float32 if np.asarray(raw).dtype == np.float32 else torch.float64)
    on_gpu = isinstance(raw, torch.Tensor) and raw.is_cuda
    blocks = []
    for x in (pressure, parcel_temperature, temperature):
        b = lay.to_block(x, None, dtype).cuda()
        if b.dim() == 1:
            b = b[:, None].expand(lay.L, int(np.prod(lay.col_shape)) if lay.col_shape else 1)
        blocks.append(b.contiguous())
    lp = lay.scalar_to_block(lcl_pressure, dtype).cuda()
    lt = lay.scalar_to_block(lcl_temperature, dtype).cuda()
    _clear_flags(ctx)
    r = ctx.lfc_el(blocks[0], blocks[1], blocks[2], lp, lt)
    _check_flags(ctx)
    fix = (lambda x: x) if on_gpu else (lambda x: x.cpu())
    return lay.dataset({k: lay.wrap_scalar(fix(v), k) for k, v in r.items()})


def cape_cin_base(pressure, temperature, lfc_pressure, el_pressure, parcel_temperature,
                  vert_dim="model_level_number", pos_cape_neg_cin=True, post_zero_cin=False,
                  vert_axis=0, device=None, **kwargs):
    """PF:1291-1392 (extra kwargs are swallowed like the reference's ``**kwargs``, PF:1293)."""
    ctx = _lib.get_context(device)
    lay = _Layout(temperature, vert_dim, vert_axis)
    raw = temperature.data if lay.is_xr else temperature
    dtype = raw.dtype if isinstance(raw, torch.Tensor) else (torch.float32 if np.asarray(raw).dtype == np.float32 else torch.float64)
    on_gpu = isinstance(raw, torch.Tensor) and raw.is_cuda
    blocks = []
    for x in (pressure, temperature, parcel_temperature):
        b = lay.to_block(x, None, dtype).cuda()
        if b.dim() == 1:
            b = b[:, None].expand(lay.L, int(np.prod(lay.col_shape)) if lay.col_shape else 1)
        blocks.append(b.contiguous())
    lf = lay.scalar_to_block(lfc_pressure, dtype).cuda()
    el = lay.scalar_to_block(el_pressure, dtype).cuda()
    opts = _lib.make_options(pos_cape_neg_cin=pos_cape_neg_cin, post_zero_cin=post_zero_cin)
    r = ctx.cape_cin_base(blocks[0], blocks[1], lf, el, blocks[2], opts)
    fix = (lambda x: x) if on_gpu else (lambda x: x.cpu())
    return lay.dataset({k: lay.wrap_scalar(fix(v), k) for k, v in r.items()})


# ---- derived convective indices (SURVEY.md 8f-1) ------------------------------------------------------
def _blocks(lay, arrays, dtype):
    """Inputs -> CUDA level-major blocks ([L, N]; a 1-D vertical axis stays [L])."""
    out = []
    for x in arrays:
        b = lay.to_block(x, None, dtype)
        out.append(b.cuda() if not b.is_cuda else b)
    return out


def _layout_of(template, vert_dim, vert_axis):
    lay = _Layout(template, vert_dim, vert_axis)
    raw = template.data if lay.is_xr else template
    if isinstance(raw, torch.Tensor):
        dtype = raw.dtype if raw.dtype in (torch.float32, torch.float64) else torch.float64
        on_gpu = raw.is_cuda
    else:
        dtype = torch.float32 if np.asarray(raw).dtype == np.float32 else torch.float64
        on_gpu = False
    return lay, dtype, on_gpu


def linear_interp(x, coords, at, dim="model_level_number", keep_attrs=True, extrapolate=False, vert_axis=0,
                  device=None, log=False):
    """PF:1758-1811 for one field ``x`` (``extrapolate=True`` is not on the parcel path and not implemented)."""
    assert not extrapolate, "extrapolate=True is not implemented"
    ctx = _lib.get_context(device)
    lay, dtype, on_gpu = _layout_of(x, dim, vert_axis)
    xb, cb = _blocks(lay, [x, coords], dtype)
    at_v = at if np.isscalar(at) else lay.scalar_to_block(at, dtype).cuda()
    (res,) = ctx.interp_levels(cb, [xb], at_v, log=log)
    return lay.wrap_scalar(res if on_gpu else res.cpu(), None)


def log_interp(x, coords, at, dim="model_level_number", vert_axis=0, device=None):
    """PF:1813-1828."""
    return linear_interp(x, coords, at, dim=dim, vert_axis=vert_axis, device=device, log=True)


def lifted_index(profile, vert_dim="model_level_number", description=None, prefix=None, vert_axis=0, device=None):
    """PF:1722-1756: environment minus parcel temperature of a parcel_profile_with_lcl() profile,
    log-interpolated to 500 hPa."""
    ctx = _lib.get_context(device)
    lay, dtype, on_gpu = _layout_of(profile["temperature"], vert_dim, vert_axis)
    tp, te, p = _blocks(lay, [profile["temperature"], profile["environment_temperature"], profile["pressure"]], dtype)
    a, b = ctx.interp_levels(p, [tp, te], 500.0, log=True)
    li = b - a
    name = "lifted_index" if prefix is None else prefix + "_lifted_index"
    ds = lay.dataset({name: lay.wrap_scalar(li if on_gpu else li.cpu(), "lifted_index")})
    attrs = {"long_name": "Lifted index", "units": "K"}
    if description is not None:
        attrs["description"] = description
    if isinstance(ds, Dataset):
        ds.var_attrs[name] = attrs
    else:
        ds[name].attrs.update(attrs)
    return ds


def deep_convective_index(pressure, temperature, dewpoint, lifted_index, vert_dim="model_level_number",
                          description=None, prefix=None, vert_axis=0, device=None):
    """PF:1830-1870 (Kunz 2009): T(850 hPa) + Td(850 hPa) [C] - lifted index."""
    ctx = _lib.get_context(device)
    lay, dtype, on_gpu = _layout_of(temperature, vert_dim, vert_axis)
    t, td, p = _blocks(lay, [temperature, dewpoint, pressure], dtype)
    a, b = ctx.interp_levels(p, [t, td], 850.0, log=True)
    li = lay.scalar_to_block(lifted_index, dtype).cuda()
    dci = (a - 273.15) + (b - 273.15) - li
    name = "dci" if prefix is None else prefix + "_dci"
    ds = lay.dataset({name: lay.wrap_scalar(dci if on_gpu else dci.cpu(), "dci")})
    attrs = {"long_name": "Deep convective index", "units": "C"}
    if description is not None:
        attrs["description"] = description
    if isinstance(ds, Dataset):
        ds.var_attrs[name] = attrs
    else:
        ds[name].attrs.update(attrs)
    return ds


def isobar_temperature(pressure, temperature, isobar, vert_dim="model_level_number", vert_axis=0, device=None):
    """PF:2193-2214: temperature log-interpolated to ``isobar`` hPa."""
    return log_interp(temperature, pressure, isobar, dim=vert_dim, vert_axis=vert_axis, device=device)


def lapse_rate(pressure, temperature, height, from_pressure=700, to_pressure=500, vert_dim="model_level_number",
               vert_axis=0, device=None):
    """PF:2102-2135: environmental lapse rate between two pressures [K/km]."""
    ctx = _lib.get_context(device)
    lay, dtype, on_gpu = _layout_of(temperature, vert_dim, vert_axis)
    t, h, p = _blocks(lay, [temperature, height, pressure], dtype)
    ft, fh = ctx.interp_levels(p, [t, h], float(from_pressure), log=True)
    tt, th = ctx.interp_levels(p, [t, h], float(to_pressure), log=True)
    lapse = (tt - ft) / (th / 1000 - fh / 1000)
    return lay.wrap_scalar(lapse if on_gpu else lapse.cpu(), None)


def freezing_level_height(temperature, height, vert_dim="model_level_number", vert_axis=0, device=None, level=273.15):
    """PF:2137-2160: lowest height at which the temperature crosses 273.15 K."""
    ctx = _lib.get_context(device)
    lay, dtype, on_gpu = _layout_of(temperature, vert_dim, vert_axis)
    t, h = _blocks(lay, [temperature, height], dtype)
    r = ctx.level_crossing(h, t, level)
    return lay.wrap_scalar(r if on_gpu else r.cpu(), None)


def wet_bulb_temperature_fast(temperature, dewpoint):
    """PF:364-387: the "1/3 rule" (Knox et al. 2017); elementwise on the caller's array library."""
    return temperature - (1 / 3) * (temperature - dewpoint)


def wet_bulb_temperature(pressure, temperature, dewpoint, vert_dim="model_level_number", device=None):
    """PF:389-445, Normand's rule: every point is lifted to its LCL (PF:609-682) and brought back down the
    moist adiabat of the lookup tables to its own pressure (``xp_wet_bulb_temperature``: one thread per
    point instead of the reference's Python loop over levels)."""
    lookup_tables_loaded(device)
    return _pointwise("wet_bulb_temperature", [pressure, temperature, dewpoint], template=1,
                      name="wet_bulb_temperature", attrs={"long_name": "Wet bulb temperature", "units": "K"},
                      device=device)


def downdraft_cape(pressure, temperature, dewpoint, vert_dim="model_level_number", vert_axis=0, metpy_compat="1.4.1",
                   profile=False, device=None):
    """Downdraft CAPE after MetPy's ``downdraft_cape``, on this library's thermodynamics and lookup-table moist
    adiabat (``xp_downdraft_cape``, one CUDA thread per column; contract in DESIGN.md section 3.12).

    The downdraft starts at the minimum equivalent potential temperature in the 700-500 hPa layer, at its wet-bulb
    temperature, and descends moist-adiabatically to the surface; ``dcape`` is -Rd times the integral of the
    environment minus parcel virtual temperature over ln p, not clipped (negative where the parcel is warmer).
    Columns that do not span 700-500 hPa give NaN.  Returns a Dataset of dcape [J/kg], downdraft_start_pressure
    [hPa] and downdraft_start_temperature [K] and, with ``profile=True``, downdraft_parcel_temperature on the input
    levels (NaN above the start and on levels with a NaN input)."""
    lookup_tables_loaded(device)
    ctx = _lib.get_context(device)
    lay, dtype, on_gpu = _layout_of(temperature, vert_dim, vert_axis)
    t, td, p = _blocks(lay, [temperature, dewpoint, pressure], dtype)
    r = ctx.downdraft_cape(p, t, td, metpy_compat=metpy_compat, profile=profile)
    fix = (lambda x: x) if on_gpu else (lambda x: x.cpu())
    out = {k: lay.wrap_scalar(fix(r[k]), k) for k in _lib.DOWNDRAFT_FIELDS}
    if profile:
        out["downdraft_parcel_temperature"] = lay.wrap_profile(fix(r["downdraft_parcel_temperature"]),
                                                               "downdraft_parcel_temperature", lay.L)
    return lay.dataset(out)


def effective_inflow_layer(pressure, temperature, dewpoint, vert_dim="model_level_number", vert_axis=0, min_cape=100,
                           min_cin=-250, most_unstable_depth=300, profile=False, device=None, **kwargs):
    """The effective inflow layer (Thompson et al. 2007, SHARPpy's ``effective_inflow_layer``) on this library's
    parcel lift (``xp_effective_inflow_layer``; contract in DESIGN.md section 3.13).

    A level is valid when pressure, temperature and dewpoint are all non-NaN.  The parcel of a valid level is lifted
    over the levels above it, with CAPE / CIN as ``cape_cin`` computes them (``kwargs``: its options,
    ``virtual_temperature_correction``, ``lcl_interp``, ``pos_cape_neg_cin``, ``post_zero_cin``, ``metpy_compat``),
    and passes when CAPE >= ``min_cape`` and CIN > ``min_cin`` [J/kg].  If the most-unstable parcel (over
    ``most_unstable_depth`` hPa) fails, the column has no layer.  Otherwise the base is the first passing level from
    the surface up and the top is the last passing level before the first failing one above it.  Returns a Dataset
    of effective_inflow_base and effective_inflow_top [hPa] (NaN: no layer) and, with ``profile=True``,
    level_parcel_cape and level_parcel_cin on the input levels (NaN on invalid levels), which lifts every valid
    level of every column."""
    lookup_tables_loaded(device)
    ctx = _lib.get_context(device)
    lay, dtype, on_gpu = _layout_of(temperature, vert_dim, vert_axis)
    dev = f"cuda:{ctx.device}"
    t, td, p = [b.to(dev).contiguous() for b in _blocks(lay, [temperature, dewpoint, pressure], dtype)]
    opts = _lib.make_options(most_unstable_depth=most_unstable_depth, **_options(kwargs))
    _clear_flags(ctx)
    r = ctx.effective_inflow_layer(p, t, td, options=opts, min_cape=min_cape, min_cin=min_cin, profile=profile)
    _check_flags(ctx)
    fix = (lambda x: x) if on_gpu else (lambda x: x.cpu())
    out = {k: lay.wrap_scalar(fix(r[k]), k) for k in _lib.EFFECTIVE_FIELDS}
    if profile:
        for k in _lib.EFFECTIVE_LEVEL_FIELDS:
            out[k] = lay.wrap_profile(fix(r[k]), k, lay.L)
    return lay.dataset(out)


def _wind_blocks(surface_wind_u, surface_wind_v, wind_u, wind_v, height, vert_dim, vert_axis, device):
    ctx = _lib.get_context(device)
    lay, dtype, on_gpu = _layout_of(wind_u, vert_dim, vert_axis)
    dev = f"cuda:{ctx.device}"
    u, v, h = [b.to(dev) for b in _blocks(lay, [wind_u, wind_v, height], dtype)]
    su, sv = [lay.scalar_to_block(x, dtype).to(dev) for x in (surface_wind_u, surface_wind_v)]
    return ctx, lay, on_gpu, h, u, v, su, sv


def bunkers_storm_motion(surface_wind_u, surface_wind_v, wind_u, wind_v, height, vert_dim="model_level_number",
                         vert_axis=0, device=None):
    """Bunkers et al. (2000) storm motion by the internal-dynamics method, on the height-weighted 0-6 km mean wind
    (``xp_storm_kinematics``, one CUDA thread per column; contract in DESIGN.md section 3.14).

    The wind profile is the surface wind at 0 m followed by the levels with non-NaN height, u and v above the surface
    (``height`` in m above the surface; levels at or below ground are dropped), linear in height.  The shear vector S is
    the 5.5-6 km mean wind minus the 0-0.5 km mean wind; the right / left movers are the 0-6 km mean wind plus / minus
    7.5 m/s normal to S.  Columns that do not reach 6 km, whose heights do not increase, with a NaN surface wind or
    with S = 0 give NaN.  Returns a Dataset of bunkers_right_u/_v, bunkers_left_u/_v and mean_wind_u/_v [m/s]."""
    ctx, lay, on_gpu, h, u, v, su, sv = _wind_blocks(surface_wind_u, surface_wind_v, wind_u, wind_v, height,
                                                     vert_dim, vert_axis, device)
    r = ctx.storm_kinematics(h, u, v, su, sv)
    fix = (lambda x: x) if on_gpu else (lambda x: x.cpu())
    return lay.dataset({k: lay.wrap_scalar(fix(r[k]), k) for k in _lib.MOTION_FIELDS})


def storm_relative_helicity(surface_wind_u, surface_wind_v, wind_u, wind_v, height, depths=(1000, 3000),
                            mover="right", vert_dim="model_level_number", vert_axis=0, device=None):
    """Storm-relative helicity over 0-d m above the surface for each of up to 4 ``depths``, relative to the Bunkers
    motion of the ``mover`` ('right' or 'left'; ``xp_storm_kinematics``, contract in DESIGN.md section 3.14).

    SRH is MetPy's ``storm_relative_helicity`` total over the layer's points (its bottom, the profile levels inside,
    its top, interpolated linearly in height), positive for a veering hodograph with the right mover.  NaN where the
    Bunkers motion is NaN or the profile does not reach the depth.  Returns a Dataset of srh_0_<d>m [m2/s2]."""
    ctx, lay, on_gpu, h, u, v, su, sv = _wind_blocks(surface_wind_u, surface_wind_v, wind_u, wind_v, height,
                                                     vert_dim, vert_axis, device)
    r = ctx.storm_kinematics(h, u, v, su, sv, mover=mover, depths=depths,
                             outputs=[f"srh_0_{float(d):g}m" for d in depths])
    fix = (lambda x: x) if on_gpu else (lambda x: x.cpu())
    attrs = {k: {"long_name": f"Storm-relative helicity, {k[6:-1]} m ({mover} mover)", "units": "m$^{2}$ s$^{-2}$"}
             for k in r}
    ds = lay.dataset({k: lay.wrap_scalar(fix(r[k]), k) for k in r})
    for k in r:
        if isinstance(ds, Dataset):
            ds.var_attrs[k] = attrs[k]
        else:
            ds[k].attrs.update(attrs[k])
    return ds


def supercell_composite_parameter(mucape, effective_srh, effective_bulk_wind_difference, device=None):
    """Supercell composite parameter, SHARPpy's ``params.scp``: (mucape / 1000) (esrh / 50) t_b with t_b = 0 below
    10 m/s of effective bulk wind difference, 1 above 20 m/s and ebwd / 20 between (``xp_supercell_tornado_parameters``,
    pointwise; NaN in gives NaN out).  Units J/kg, m2/s2, m/s."""
    return _pointwise("supercell_composite_parameter", [mucape, effective_srh, effective_bulk_wind_difference],
                      name="supercell_composite_parameter", attrs=_ATTRS["supercell_composite_parameter"],
                      device=device)


def significant_tornado_parameter(mlcape, effective_srh, effective_bulk_wind_difference, lcl_height, mlcin,
                                  device=None):
    """Effective-layer significant tornado parameter with CIN, SHARPpy's ``params.stp_cin``: max(0, (mlcape / 1500)
    (esrh / 150) t_b t_lcl t_cin) with t_b = 0 below 12.5 m/s of effective bulk wind difference, 1.5 above 30 m/s and
    ebwd / 20 between; t_lcl = 1 below 1000 m of mixed-layer LCL height above the surface, 0 above 2000 m and
    (2000 - lcl) / 1000 between; t_cin = 1 above -50 J/kg of mixed-layer CIN, 0 below -200 and (cin + 200) / 150 between
    (``xp_supercell_tornado_parameters``, pointwise; NaN in gives NaN out)."""
    return _pointwise("significant_tornado_parameter", [mlcape, effective_srh, effective_bulk_wind_difference,
                                                        lcl_height, mlcin],
                      name="significant_tornado_parameter", attrs=_ATTRS["significant_tornado_parameter"],
                      device=device)


def effective_layer_parameters(pressure, temperature, dewpoint, height, wind_u, wind_v, surface_wind_u,
                               surface_wind_v, mover="right", min_cape=100, min_cin=-250, most_unstable_depth=300,
                               mixed_layer_depth=100, vert_dim="model_level_number", vert_axis=0, device=None,
                               **kwargs):
    """Effective storm-relative helicity (ESRH), effective bulk wind difference (EBWD), the supercell composite
    parameter and the effective-layer significant tornado parameter (contract in DESIGN.md section 3.14).

    The effective inflow layer is ``effective_inflow_layer``'s (``min_cape``, ``min_cin``, ``most_unstable_depth`` and
    ``kwargs``, cape_cin's options); one lift gives the mixed-layer (``mixed_layer_depth`` hPa) and most-unstable
    (``most_unstable_depth`` hPa) parcels.  ``height`` is m above the surface on the levels of ``pressure``; the
    heights of the layer's base and top, the MU equilibrium level and the ML LCL are ``log_interp`` of it.  ESRH is
    the SRH of the ``mover``'s Bunkers motion over the layer; EBWD is the bulk wind difference from the base (at least
    the surface) up to half the MU EL height above it.  Columns without an effective layer have NaN ESRH and EBWD and
    enter the composites with ESRH = EBWD = 0 (so SCP and STP are 0 there unless another input is NaN); for
    ``mover='left'`` the composites take -ESRH.  Returns a Dataset of effective_inflow_base / _top [hPa],
    effective_srh [m2/s2], effective_bulk_wind_difference [m/s], supercell_composite_parameter and
    significant_tornado_parameter."""
    lookup_tables_loaded(device)
    ctx = _lib.get_context(device)
    lay, dtype, on_gpu = _layout_of(temperature, vert_dim, vert_axis)
    dev = f"cuda:{ctx.device}"
    t, td, p = [b.to(dev).contiguous() for b in _blocks(lay, [temperature, dewpoint, pressure], dtype)]
    u, v, h = [b.to(dev) for b in _blocks(lay, [wind_u, wind_v, height], dtype)]
    su, sv = [lay.scalar_to_block(x, dtype).to(dev) for x in (surface_wind_u, surface_wind_v)]
    opt = _options(kwargs)
    _clear_flags(ctx)
    eff = ctx.effective_inflow_layer(p, t, td, options=_lib.make_options(most_unstable_depth=most_unstable_depth, **opt),
                                     min_cape=min_cape, min_cin=min_cin)
    lifted = ctx.cape_cin(p, t, td, kinds=("ml", "mu"), options=_lib.make_options(
        mixed_layer_depth=mixed_layer_depth, most_unstable_depth=most_unstable_depth, **opt))
    _check_flags(ctx)
    base, top = eff["effective_inflow_base"], eff["effective_inflow_top"]
    ml, mu = lifted["ml"], lifted["mu"]
    hc = h.contiguous()
    (z_base,), (z_top,), (z_el,), (z_lcl,) = [ctx.interp_levels(p, [hc], x, log=True)
                                              for x in (base, top, mu["el_pressure"], ml["lcl_pressure"])]
    zb0 = torch.clamp(z_base, min=0.0)                               # NaN stays NaN, like np.maximum
    kin = ctx.storm_kinematics(h, u, v, su, sv, mover=mover, srh_layer=(z_base, z_top),
                               bwd_layer=(zb0, zb0 + (z_el - zb0) / 2.0),
                               outputs=["srh_layer", "bulk_wind_difference"])
    no_layer = torch.isnan(base)
    esrh = torch.where(no_layer, torch.full_like(base, float("nan")), kin["srh_layer"])
    ebwd = torch.where(no_layer, torch.full_like(base, float("nan")), kin["bulk_wind_difference"])
    s_in = torch.where(no_layer, torch.zeros_like(esrh), esrh) * _lib.MOVERS[mover]
    b_in = torch.where(no_layer, torch.zeros_like(ebwd), ebwd)
    comp = ctx.supercell_tornado_parameters(mu["cape"], s_in, b_in, ml["cape"], ml["cin"], z_lcl)
    fix = (lambda x: x) if on_gpu else (lambda x: x.cpu())
    out = {"effective_inflow_base": base, "effective_inflow_top": top, "effective_srh": esrh,
           "effective_bulk_wind_difference": ebwd}
    out.update(comp)
    return lay.dataset({k: lay.wrap_scalar(fix(x), k) for k, x in out.items()})


def _vertical_pressure(pressure, lay):
    """A shared 1-D pressure axis [L] reshaped to broadcast along the layout's vertical axis.  The pointwise functions
    broadcast like NumPy, which would align [L] with the last axis of the fields instead; anything else (per-point
    pressure, xarray inputs, which align by dimension name) is returned as it is."""
    if lay.is_xr or len(lay.shape) < 2 or lay.vert_axis is None:
        return pressure
    if not isinstance(pressure, torch.Tensor):
        pressure = np.asarray(pressure)
    if pressure.ndim != 1 or pressure.shape[0] != lay.L:
        return pressure
    shape = [1] * len(lay.shape)
    shape[lay.vert_axis] = lay.L
    return pressure.reshape(shape)


def melting_level_height(pressure, temperature, dewpoint, height, fast=True, vert_dim="model_level_number",
                         vert_axis=0, device=None):
    """PF:2162-2191: lowest height at which the wet-bulb temperature (1/3 rule with fast=True, Normand's
    rule otherwise) crosses 273.15 K.  Returns (melting level height, wet bulb)."""
    if fast:
        wb = wet_bulb_temperature_fast(temperature, dewpoint)
    else:
        p = _vertical_pressure(pressure, _Layout(temperature, vert_dim, vert_axis))
        wb = wet_bulb_temperature(p, temperature, dewpoint, vert_dim=vert_dim, device=device)
    return freezing_level_height(wb, height, vert_dim=vert_dim, vert_axis=vert_axis, device=device), wb


def wind_shear(surface_wind_u, surface_wind_v, wind_u, wind_v, height, shear_height=6000,
               vert_dim="model_level_number", vert_axis=0, device=None):
    """PF:2216-2259: wind at ``shear_height`` (linear in height) minus the surface wind."""
    ctx = _lib.get_context(device)
    lay, dtype, on_gpu = _layout_of(wind_u, vert_dim, vert_axis)
    u, v, h = _blocks(lay, [wind_u, wind_v, height], dtype)
    hu, hv = ctx.interp_levels(h, [u, v], float(shear_height), log=False)
    su = lay.scalar_to_block(surface_wind_u, dtype).cuda()
    sv = lay.scalar_to_block(surface_wind_v, dtype).cuda()
    shear_u, shear_v = hu - su, hv - sv
    out = {"shear_u": shear_u, "shear_v": shear_v,
           "shear_magnitude": torch.sqrt(shear_u ** 2 + shear_v ** 2),
           "positive_shear": torch.sqrt(hu ** 2 + hv ** 2) > torch.sqrt(su ** 2 + sv ** 2)}
    return lay.dataset({k: lay.wrap_scalar(x if on_gpu else x.cpu(), None) for k, x in out.items()})


def dewpoint_from_specific_humidity(pressure, temperature, specific_humidity, metpy_compat="1.4.1", device=None):
    """metpy.calc.dewpoint_from_specific_humidity as the reference calls it (PF:1889, 1969), on the GPU
    (``xp_dewpoint_from_specific_humidity``).  MetPy 1.4.1 goes through relative humidity, MetPy >= 1.6 through
    the vapour pressure (environment_changes_eval.ipynb:278) -- pass the version the data were made with."""
    return _pointwise("dewpoint_from_specific_humidity", [pressure, temperature, specific_humidity], template=1,
                      name="dewpoint", attrs={"long_name": "Dewpoint temperature", "units": "K"}, device=device,
                      metpy_compat=str(metpy_compat))


def significant_hail_parameter(mucape, mixing_ratio, lapse, temp_500, shear, flh, device=None):
    """PF:2261-2306 (https://www.spc.noaa.gov/exper/mesoanalysis/help/help_sigh.html): MU CAPE [J/kg], MU parcel
    mixing ratio [kg/kg], 700-500 hPa lapse rate [K/km], 500 hPa temperature [K], 0-6 km shear [m/s],
    freezing level height [m]  (``xp_significant_hail_parameter``)."""
    return _pointwise("significant_hail_parameter", [mucape, mixing_ratio, lapse, temp_500, shear, flh],
                      name="ship", attrs={"long_name": "Significant hail parameter",
                                          "units": "J kg$^{-2}$ g K$^2$ km$^{-1}$ m s$^{-1}$"}, device=device)


_PROXY_NAMES = {"proxy_Craven2004": "Craven 2004", "proxy_Kunz2007": "Kunz 2007", "proxy_Trapp2007": "Trapp 2007",
                "proxy_Marsh2009": "Marsh 2009", "proxy_Allen2011": "Allen 2011", "proxy_Allen2014": "Allen 2014",
                "proxy_Eccel2012": "Eccel 2012", "proxy_Mohr2013": "Mohr 2013", "proxy_SHIP_0.1": "SHIP > 0.1"}


def storm_proxies(dat, device=None):
    """PF:2323-2407: the nine storm proxies (True = triggered) and SHIP from the variables ``conv_properties``
    returns (``xp_storm_proxies``, one thread per column)."""
    ctx = _lib.get_context(device)
    names = {k: ("shear_magnitude" if k == "shear_magnitude" else k) for k in _lib.PROXY_INPUTS}
    raw = {k: dat[names[k]] for k in _lib.PROXY_INPUTS}
    tmpl = raw["mixed_100_cape"]
    is_xr = _xr is not None and isinstance(tmpl, _xr.DataArray)
    if is_xr:
        xa = _xr.broadcast(*[raw[k] for k in _lib.PROXY_INPUTS])
        tmpl = xa[0]
        raw = {k: a.data for k, a in zip(_lib.PROXY_INPUTS, xa)}
    src = raw["mixed_100_cape"]
    if isinstance(src, torch.Tensor):
        dt = src.dtype if src.dtype in (torch.float32, torch.float64) else torch.float64
    else:
        dt = torch.float32 if np.asarray(src).dtype == np.float32 else torch.float64
    dev = {}
    for k, v in raw.items():
        if isinstance(v, torch.Tensor):
            dev[k] = v.to(dt).cuda()
        else:
            dev[k] = torch.as_tensor(np.asarray(v).astype(np.float64)).to(dt).cuda()
    res = ctx.storm_proxies(dev)
    out = {}
    for k, v in res.items():
        if is_xr:
            da = tmpl.copy(data=v.cpu().numpy())
            da.attrs = {}
            da.name = k
            out[k] = da
        elif isinstance(src, torch.Tensor):
            out[k] = v if src.is_cuda else v.cpu()
        else:
            out[k] = v.cpu().numpy()
    if is_xr:
        ds = _xr.Dataset(out)
        for k, val in _PROXY_NAMES.items():
            ds[k].attrs["long_name"] = "Proxy " + val
        ds["ship"].attrs["long_name"] = "Significant hail parameter (SHIP)"
        ds["ship"].attrs["units"] = "J kg$^{-2}$ g K$^2$ km$^{-1}$ m s$^{-1}$"
        return ds
    ds = Dataset(out)
    ds.var_attrs = {k: {"long_name": "Proxy " + val} for k, val in _PROXY_NAMES.items()}
    ds.var_attrs["ship"] = {"long_name": "Significant hail parameter (SHIP)",
                            "units": "J kg$^{-2}$ g K$^2$ km$^{-1}$ m s$^{-1}$"}
    return ds


def _conv(dat, vert_dim, vert_axis, device, min_set, ignore_nans, metpy_compat, downdraft=False, effective=False,
          kinematics=False, mover="right"):
    p, t = dat["pressure"], dat["temperature"]
    td = dewpoint_from_specific_humidity(_vertical_pressure(p, _Layout(t, vert_dim, vert_axis)), t,
                                         dat["specific_humidity"], metpy_compat, device=device)
    try:
        dat["dewpoint"] = td                                        # the reference adds it to the caller's Dataset
    except Exception:
        pass
    kw = dict(vert_dim=vert_dim, vert_axis=vert_axis, device=device)
    out = {}
    # the lifting kernels read (p, T, q) themselves and convert q in their load stage (xp_columns.
    # dewpoint_is_specific_humidity); `td` above is only what the reference hands back / what the indices need
    q = dat["specific_humidity"]
    lift = dict(kw, metpy_compat=metpy_compat, specific_humidity=True)

    def merge(ds):
        for k in ds:
            out[k] = ds[k]

    def parcel_block(prefix, cc, prof, desc):
        merge(cc)
        li = lifted_index(prof, prefix=prefix, description="Lifted index using " + desc, **kw)
        merge(li)
        if not min_set:
            merge(deep_convective_index(p, t, td, li[prefix + "_lifted_index"], prefix=prefix,
                                        description="Deep convective index using " + desc, **kw))

    if not min_set:
        cc, prof, mu_parcel = most_unstable_cape_cin(p, t, q, depth=250, prefix="mu", **lift)
        parcel_block("mu", cc, prof, "most-unstable parcel in lowest 250 hPa.")
        out["mu_mixing_ratio"] = _pointwise("saturation_mixing_ratio", [mu_parcel["pressure"], mu_parcel["dewpoint"]],
                                            name="mu_mixing_ratio", device=device)   # PF:2047-2053
    cc, prof, _ = mixed_layer_cape_cin(p, t, q, depth=100, prefix="mixed_100", **lift)
    parcel_block("mixed_100", cc, prof, "fully-mixed lowest 100 hPa parcel.")
    if not min_set:
        cc, prof, _ = mixed_layer_cape_cin(p, t, q, depth=50, prefix="mixed_50", **lift)
        parcel_block("mixed_50", cc, prof, "fully-mixed lowest 50 hPa parcel.")
    out["lapse_rate_700_500"] = lapse_rate(p, t, dat["height_asl"], **kw)
    out["temp_500"] = isobar_temperature(p, t, 500, **kw)
    out["freezing_level"] = freezing_level_height(t, dat["height_asl"], **kw)
    out["melting_level"], _ = melting_level_height(p, t, td, dat["height_asl"], **kw)
    merge(wind_shear(dat["surface_wind_u"], dat["surface_wind_v"], dat["wind_u"], dat["wind_v"],
                     dat["wind_height_above_surface"], shear_height=6000, **kw))
    if downdraft:
        out["dcape"] = downdraft_cape(p, t, td, metpy_compat=metpy_compat, **kw)["dcape"]
    winds = (dat["surface_wind_u"], dat["surface_wind_v"], dat["wind_u"], dat["wind_v"], dat["wind_height_above_surface"])
    if kinematics:
        merge(bunkers_storm_motion(*winds, **kw))
        merge(storm_relative_helicity(*winds, depths=(1000, 3000), mover=mover, **kw))
    if effective and kinematics:
        merge(effective_layer_parameters(p, t, td, winds[4], winds[2], winds[3], winds[0], winds[1], mover=mover,
                                         metpy_compat=metpy_compat, **kw))
    elif effective:
        eff = effective_inflow_layer(p, t, td, metpy_compat=metpy_compat, **kw)
        for k in _lib.EFFECTIVE_FIELDS:
            out[k] = eff[k]
    if not min_set and not ignore_nans:                              # PF:1976-1983, 2098-2099
        lay = _Layout(t, vert_dim, vert_axis)
        va = lay.vert_axis if lay.vert_axis is not None else 0
        if lay.is_xr:
            bad = (np.isnan(td).any(vert_dim) | np.isnan(p).any(vert_dim) | np.isnan(t).any(vert_dim) |
                   np.isnan(dat["specific_humidity"]).any(vert_dim))
            out = {k: v.where(~bad) for k, v in out.items()}
        else:
            lib = torch if isinstance(t, torch.Tensor) else np
            bad = None
            for x in (td, p, t, dat["specific_humidity"]):
                b = lib.isnan(x).any(va) if x.ndim > 1 else lib.isnan(x).any()
                bad = b if bad is None else (bad | b)
            def mask(v):
                if lib is torch:
                    v = v.to(torch.float64) if v.dtype == torch.bool else v
                    b = bad.to(v.device) if isinstance(bad, torch.Tensor) else bad
                    return torch.where(b, torch.full_like(v, float("nan")), v)
                v = v.astype(np.float64) if v.dtype == np.bool_ else v
                return np.where(bad, np.nan, v)

            out = {k: mask(v) for k, v in out.items()}
    lay = _Layout(t, vert_dim, vert_axis)
    return lay.dataset(out)


def conv_properties(dat, vert_dim="model_level_number", ignore_nans=False, vert_axis=0, device=None,
                    metpy_compat="1.4.1", downdraft=False, effective=False, kinematics=False, mover="right"):
    """PF:1951-2100: MU (250 hPa) and mixed (100, 50 hPa) CAPE/CIN, lifted and deep-convective indices,
    MU mixing ratio, 700-500 hPa lapse rate, 500 hPa temperature, freezing/melting level, 0-6 km shear.
    ``dat``: Dataset/dict with pressure, temperature, specific_humidity, height_asl, wind_u, wind_v,
    wind_height_above_surface (all [level, ...]) and surface_wind_u, surface_wind_v.  ``downdraft=True`` adds
    ``dcape`` (``downdraft_cape`` on the dewpoint derived from the specific humidity), masked like the rest;
    ``effective=True`` adds ``effective_inflow_base`` and ``effective_inflow_top`` (``effective_inflow_layer`` with
    its defaults on that dewpoint), masked the same way.  ``kinematics=True`` adds the Bunkers storm motion
    (``bunkers_storm_motion``: bunkers_right_u/_v, bunkers_left_u/_v, mean_wind_u/_v) and srh_0_1000m / srh_0_3000m
    (``storm_relative_helicity`` for ``mover``) on wind_height_above_surface and the surface wind; with
    ``effective=True`` as well it adds effective_srh, effective_bulk_wind_difference, supercell_composite_parameter and
    significant_tornado_parameter from one ``effective_layer_parameters`` call, whose base and top are the
    effective_inflow_base / _top it returns.  All are masked like the rest."""
    return _conv(dat, vert_dim, vert_axis, device, False, ignore_nans, metpy_compat, downdraft, effective, kinematics,
                 mover)


def min_conv_properties(dat, vert_dim="model_level_number", vert_axis=0, device=None, metpy_compat="1.4.1"):
    """PF:1872-1949: the minimal set (mixed-100 CAPE/CIN + lifted index, lapse rate, T500, freezing and
    melting level, shear)."""
    return _conv(dat, vert_dim, vert_axis, device, True, True, metpy_compat)
