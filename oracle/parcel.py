"""NumPy restatement of the reference's parcel path (whole-array, float64).

TEST INFRASTRUCTURE (see ``oracle/__init__.py``).

Every function follows the function of the same name in
``/root/reference/modules/parcel_functions.py`` ("PF"), operation by operation,
with xarray's labelled semantics (``where``/``shift``/``diff``/``rolling``/
inner-join alignment / NaN-skipping reductions) spelled out on plain arrays.

Array convention: the vertical dimension is axis 0 ("level-major"), every other
dimension is flattened into axis 1: shape ``[L, N]``.  Per-column quantities
have shape ``[N]``.  A "dataset" is a dict of such arrays.

The moist adiabat is pluggable (PF:525 is monkey-patched the same way by the
reference's own tests, unit_tests.py:114-140 / parcel_functions_demo.ipynb
cell 33): ``MoistLapseODE`` (exact, used for the MetPy-derived known answers)
or ``MoistLapseLUT`` (the reference's production lookup table, PF:525-607).
"""

import warnings

import numpy as np

from . import thermo as th

FILL = -999


# --------------------------------------------------------------------------- helpers
def _as2d(a, n_cols=None):
    a = np.asarray(a, dtype=np.float64)
    if a.ndim == 1:
        a = a[:, None]
    if n_cols is not None and a.shape[1] != n_cols:
        a = np.broadcast_to(a, (a.shape[0], n_cols))
    return a


def _quiet(fn, *a, **k):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        with np.errstate(all="ignore"):
            return fn(*a, **k)


def nanmax(a, axis=0):
    """xarray ``.max(dim)``: skips NaN, all-NaN -> NaN."""
    return _quiet(np.nanmax, a, axis=axis) if a.shape[axis] else np.full(a.shape[1:], np.nan)


def nanmin(a, axis=0):
    return _quiet(np.nanmin, a, axis=axis) if a.shape[axis] else np.full(a.shape[1:], np.nan)


def nansum(a, axis=0):
    """xarray ``.sum(dim)``: skips NaN, all-NaN -> 0."""
    return np.nansum(a, axis=axis)


def nanmean(a, axis=0):
    return _quiet(np.nanmean, a, axis=axis)


def where(cond, a, other=np.nan):
    return np.where(cond, a, other)


# --------------------------------------------------------------------------- moist lapse
class MoistLapseODE:
    """Exact pseudo-adiabat per column (MetPy's moist_lapse; unit_tests.py:114-140)."""

    def __init__(self, solver="lsoda-tight"):
        self.solver = solver

    def __call__(self, pressure, parcel_temperature, parcel_pressure):
        pressure = _as2d(pressure)
        L, N = pressure.shape
        t0 = np.broadcast_to(np.asarray(parcel_temperature, dtype=np.float64), (N,))
        p0 = np.broadcast_to(np.asarray(parcel_pressure, dtype=np.float64), (N,))
        out = np.full((L, N), np.nan)
        for c in range(N):
            out[:, c] = th.moist_lapse_ode(pressure[:, c], t0[c], p0[c], solver=self.solver)
        return out


class MoistLapseLUT:
    """PF:525-607 ``moist_lapse`` on the two lookup tables of PF:447-523.

    ``tables`` is an ``oracle.tables.AdiabatTables`` (index grid + curves + grids).
    """

    def __init__(self, tables):
        self.tables = tables

    def __call__(self, pressure, parcel_temperature, parcel_pressure):
        tb = self.tables
        pressure = _as2d(pressure)
        L, N = pressure.shape
        t0 = np.broadcast_to(np.asarray(parcel_temperature, dtype=np.float64), (N,))
        p0 = np.broadcast_to(np.asarray(parcel_pressure, dtype=np.float64), (N,))

        # PF:554-557  .sel(pressure=..., temperature=..., method='nearest')
        ok = np.isfinite(t0) & np.isfinite(p0)
        ip = tb.nearest_pressure_index(np.where(ok, p0, tb.pressure_desc[0]))
        it = tb.nearest_temperature_index(np.where(ok, t0, tb.temperature[0]))
        adiabat_idx = tb.index_grid[ip, it].astype(np.int64)      # 0 == "no adiabat" (NaN)
        # PF:570-582: missing -> index 1 for the gather, masked back to NaN afterwards.
        valid = (adiabat_idx > 0) & ok
        gather = np.where(valid, adiabat_idx, 1) - 1               # adiabat numbers are 1-based

        # PF:585-592  np.interp(at=pressure[column], xp=P ascending, fp=curve[adiabat])
        xp = tb.pressure_asc
        out = np.full((L, N), np.nan)
        # chunk so the gathered curves (N x 2196) stay small, as dask would.
        step = 4096
        for s in range(0, N, step):
            e = min(N, s + step)
            curves = tb.curves_asc[gather[s:e]].astype(np.float64)  # [n, nP]
            at = pressure[:, s:e]
            j = np.searchsorted(xp, np.where(np.isfinite(at), at, xp[0]), side="right") - 1
            j = np.clip(j, 0, xp.size - 1)
            j1 = np.minimum(j + 1, xp.size - 1)
            cols = np.arange(e - s)[None, :]
            f0 = curves[cols, j]
            f1 = curves[cols, j1]
            with np.errstate(all="ignore"):
                slope = (f1 - f0) / (xp[j1] - xp[j])
                res = slope * (at - xp[j]) + f0
            # numpy.interp: exact node hits and the last node return fp[j] itself.
            res = np.where((xp[j] == at) | (j == xp.size - 1), f0, res)
            res = np.where(valid[s:e][None, :], res, np.nan)       # PF:582
            out[:, s:e] = res
        # PF:598-605
        out = np.where(pressure >= xp.min(), out, np.nan)
        out = np.where(pressure <= xp.max(), out, np.nan)
        out = np.where(np.isnan(t0)[None, :], np.nan, out)
        out = np.where(np.isnan(p0)[None, :], np.nan, out)
        out = np.where(np.isnan(pressure), np.nan, out)
        return out


# --------------------------------------------------------------------------- options
class Options:
    """Function kwargs of the reference that select behaviour (SURVEY.md section 5)."""

    def __init__(self, moist_lapse, metpy_compat=th.METPY_COMPAT_DEFAULT, lcl_mode="converged"):
        self.moist_lapse = moist_lapse
        self.metpy_compat = metpy_compat
        self.lcl_mode = lcl_mode


# --------------------------------------------------------------------------- PF:609-710
def mixing_ratio(temperature, dewpoint, pressure, opts):
    """PF:684-710."""
    return th.mixing_ratio_from_t_td(temperature, dewpoint, pressure, opts.metpy_compat)


def lcl(parcel_pressure, parcel_temperature, parcel_dewpoint, opts):
    """PF:609-682.  Returns dict(lcl_pressure, lcl_temperature, lcl_virtual_temperature) [N]."""
    pp = np.asarray(parcel_pressure, dtype=np.float64)
    pt = np.asarray(parcel_temperature, dtype=np.float64)
    pd_ = np.asarray(parcel_dewpoint, dtype=np.float64)
    pp, pt, pd_ = np.broadcast_arrays(pp, pt, pd_)
    valid = ~(np.isnan(pp) | np.isnan(pt) | np.isnan(pd_))           # PF:627-629
    pp = np.where(valid, pp, 1000.0)                                 # PF:632-634
    pt = np.where(valid, pt, 273.15)
    pd_ = np.where(valid, pd_, 273.15)
    press_lcl, temp_lcl = th.lcl(pp, pt, pd_, mode=opts.lcl_mode)    # PF:644
    w = mixing_ratio(temp_lcl, temp_lcl, press_lcl, opts)            # PF:653-655
    tv = th.virtual_temperature(temp_lcl, w)                         # PF:656-657
    return {"lcl_pressure": np.where(valid, press_lcl, np.nan),      # PF:680
            "lcl_temperature": np.where(valid, temp_lcl, np.nan),
            "lcl_virtual_temperature": np.where(valid, tv, np.nan)}


# --------------------------------------------------------------------------- PF:712-780
def parcel_profile(pressure, parcel_pressure, parcel_temperature, parcel_dewpoint, opts):
    """PF:712-780.  dict(pressure, temperature, virtual_temperature [L,N], lcl_* [N])."""
    pressure = _as2d(pressure)
    L, N = pressure.shape
    pp = np.broadcast_to(np.asarray(parcel_pressure, dtype=np.float64), (N,))
    pt = np.broadcast_to(np.asarray(parcel_temperature, dtype=np.float64), (N,))
    pd_ = np.broadcast_to(np.asarray(parcel_dewpoint, dtype=np.float64), (N,))
    out = {"pressure": pressure}
    out.update(lcl(pp, pt, pd_, opts))                                           # PF:736
    below_lcl = th.dry_lapse(pressure, pt[None, :], pp[None, :])                 # PF:742
    parcel_mixing_ratio = mixing_ratio(pt, pd_, pp, opts)                        # PF:748
    above_lcl = opts.moist_lapse(pressure, out["lcl_temperature"], out["lcl_pressure"])  # PF:754
    mixing_ratios = th.saturation_mixing_ratio(pressure, above_lcl)              # PF:760
    with np.errstate(invalid="ignore"):
        ge = pressure >= out["lcl_pressure"][None, :]
        le = pressure <= out["lcl_pressure"][None, :]
    out["temperature"] = np.where(ge, below_lcl, above_lcl)                      # PF:767
    mixing_ratios = np.where(le, mixing_ratios, parcel_mixing_ratio[None, :])    # PF:773
    out["virtual_temperature"] = th.virtual_temperature(out["temperature"], mixing_ratios)
    return out


# --------------------------------------------------------------------------- PF:933-990
def insert_level(d, level, coords):
    """PF:933-990.  ``d``: dict of [L,N]; ``level``: dict of [N] (its keys are kept).

    Value-based split (>= below / < above), existing coordinate kept *below* the new
    level; NaN coordinates go through the -999 fill like the reference's.
    """
    c = d[coords]
    L, N = c.shape
    assert not np.any(c == FILL), "dataset d contains fill_value."              # PF:962
    nanc = np.isnan(c)
    d = {k: np.where(nanc, float(FILL), v) for k, v in d.items()}               # PF:963
    c = d[coords]
    lev_c = np.asarray(level[coords], dtype=np.float64)[None, :]
    with np.errstate(invalid="ignore"):
        below_m = c >= lev_c                                                    # PF:965
        above_m = c < lev_c                                                     # PF:966
    out = {}
    keys = list(level.keys())                                                   # PF:984
    below_c = np.full((L + 1, N), np.nan)
    below_c[:L] = np.where(below_m, c, np.nan)
    for k in keys:
        v = d[k]
        bel = np.full((L + 1, N), np.nan)
        bel[:L] = np.where(below_m, v, np.nan)
        abv = np.full((L + 1, N), np.nan)
        abv[1:] = np.where(above_m, v, np.nan)                                  # PF:970
        out[k] = np.where(np.isnan(below_c), abv, bel)                          # PF:977
    out_c = out[coords]
    hole = np.isnan(out_c)
    for k in keys:
        new = np.broadcast_to(np.asarray(level[k], dtype=np.float64)[None, :], (L + 1, N))
        o = np.where(hole, new, out[k])                                         # PF:985
        out[k] = np.where(o != FILL, o, np.nan)                                 # PF:988
    return out


# --------------------------------------------------------------------------- PF:1758-1828
def linear_interp(x, coords, at):
    """PF:1758-1811 (extrapolate=False).  ``x``: dict of [L,N]; coords [L,N]; at [N]."""
    at = np.asarray(at, dtype=np.float64)[None, :]
    with np.errstate(invalid="ignore"):
        coords_before = nanmin(np.where(coords >= at, coords, np.nan))          # PF:1774
        coords_after = nanmax(np.where(coords <= at, coords, np.nan))           # PF:1775
    res = {}
    for k, v in x.items():
        x_before = nanmean(np.where(coords == coords_before[None, :], v, np.nan))  # PF:1798
        x_after = nanmean(np.where(coords == coords_after[None, :], v, np.nan))    # PF:1799
        with np.errstate(all="ignore"):
            r = x_before + (x_after - x_before) * ((at[0] - coords_before) /
                                                   (coords_after - coords_before))  # PF:1802
        res[k] = np.where(x_before == x_after, x_before, r)                     # PF:1806
    return res


def log_interp(x, coords, at):
    """PF:1813-1828."""
    with np.errstate(all="ignore"):
        return linear_interp(x, np.log(coords), np.log(np.asarray(at, dtype=np.float64)))


# --------------------------------------------------------------------------- PF:806-931
def add_lcl_to_profile(profile, environment, interpolator, opts):
    """PF:858-931."""
    assert interpolator in ["linear", "log"], "interpolator must be linear or log"
    level = {"pressure": profile["lcl_pressure"],
             "temperature": profile["lcl_temperature"],
             "virtual_temperature": profile["lcl_virtual_temperature"]}
    prof_lv = {k: profile[k] for k in ("pressure", "temperature", "virtual_temperature")}
    out = insert_level(prof_lv, level, "pressure")                              # PF:884
    for k in ("lcl_pressure", "lcl_temperature", "lcl_virtual_temperature"):
        out[k] = profile[k]
    if environment is not None:
        interp = linear_interp if interpolator == "linear" else log_interp
        interp_level = interp(environment, environment["pressure"], level["pressure"])
        interp_level["pressure"] = level["pressure"]                            # PF:909
        if "virtual_temperature" in interp_level:                               # PF:911-920
            mr = mixing_ratio(interp_level["temperature"], interp_level["dewpoint"],
                              interp_level["pressure"], opts)
            interp_level["virtual_temperature"] = th.virtual_temperature(
                interp_level["temperature"], mr)
        new_env = insert_level(environment, interp_level, "pressure")           # PF:923
        for k in environment:
            if k != "pressure":
                out["environment_" + k] = new_env[k]
    return out


def parcel_profile_with_lcl(pressure, temperature, dewpoint, parcel_pressure,
                            parcel_temperature, parcel_dewpoint, opts, lcl_interp="log"):
    """PF:806-856."""
    pressure = _as2d(pressure)
    N = pressure.shape[1]
    temperature = _as2d(temperature, N)
    dewpoint = _as2d(dewpoint, N)
    profile = parcel_profile(pressure, parcel_pressure, parcel_temperature, parcel_dewpoint, opts)
    mr = mixing_ratio(temperature, dewpoint, pressure, opts)                    # PF:839
    vt = th.virtual_temperature(temperature, mr)                                # PF:842
    environment = {"temperature": temperature, "virtual_temperature": vt,
                   "dewpoint": dewpoint, "pressure": profile["pressure"]}
    return add_lcl_to_profile(profile, environment, lcl_interp, opts)


# --------------------------------------------------------------------------- PF:992-1064
def find_intersections(x, a, b, log_x=False):
    """PF:992-1064.  Inputs [M,N]; outputs indexed by the *upper* level of each interval:
    arrays [M-1,N] whose row r is the reference's offset_dim label r+1."""
    with np.errstate(all="ignore"):
        if log_x:
            x = np.log(x)
        diffs = np.diff(np.sign(a - b), axis=0)                                 # PF:1019
        after = np.where(diffs == 0, 0.0, 1.0)                                  # PF:1022 (NaN -> 1)
        hit = after == 1
        sign_change = np.where(hit, np.sign(a[1:] - b[1:]), np.nan)             # PF:1030
        x0 = np.where(hit, x[:-1], np.nan)                                      # PF:1033
        x1 = np.where(hit, x[1:], np.nan)
        a0 = np.where(hit, a[:-1], np.nan)
        a1 = np.where(hit, a[1:], np.nan)
        b0 = np.where(hit, b[:-1], np.nan)
        b1 = np.where(hit, b[1:], np.nan)
        dy0 = a0 - b0
        dy1 = a1 - b1
        ix = (dy1 * x0 - dy0 * x1) / (dy1 - dy0)                                # PF:1046
        iy = ((ix - x0) / (x1 - x0)) * (a1 - a0) + a0                           # PF:1050
        if log_x:
            ix = np.exp(ix)
        return {"all_intersect_x": ix, "all_intersect_y": iy,
                "increasing_x": np.where(sign_change > 0, ix, np.nan),
                "increasing_y": np.where(sign_change > 0, iy, np.nan),
                "decreasing_x": np.where(sign_change < 0, ix, np.nan),
                "decreasing_y": np.where(sign_change < 0, iy, np.nan)}


# --------------------------------------------------------------------------- PF:1066-1198
class ReferenceAssertion(AssertionError):
    """An ``assert`` of the reference fired (same message)."""


def lfc_el(pressure, parcel_temperature, temperature, lcl_pressure, lcl_temperature):
    """PF:1066-1198.  Returns dict(lfc_pressure, lfc_temperature, el_pressure, el_temperature)."""
    pressure = _as2d(pressure)
    M, N = pressure.shape
    a = _as2d(parcel_temperature, N)
    b = _as2d(temperature, N)
    lcl_p = np.broadcast_to(np.asarray(lcl_pressure, dtype=np.float64), (N,))
    lcl_t = np.broadcast_to(np.asarray(lcl_temperature, dtype=np.float64), (N,))

    inter = find_intersections(pressure, a, b, log_x=True)                      # PF:1101
    ia = find_intersections(pressure[1:], a[1:], b[1:], log_x=True)             # PF:1108
    # .reindex_like(intersections): label 1 (row 0) missing -> NaN
    above = {k: np.concatenate([np.full((1, N), np.nan), v], axis=0) if M > 1 else v
             for k, v in ia.items()}
    if M == 1:
        above = {k: np.full((0, N), np.nan) for k in inter}
    with np.errstate(invalid="ignore"):
        use_all = b[0] != a[0]                                                  # PF:1117-1120
    inter = {k: np.where(use_all[None, :], inter[k], above[k]) for k in inter}

    with np.errstate(invalid="ignore"):
        above_lcl = inter["increasing_x"] < lcl_p[None, :]                      # PF:1127
    lfc_p = nanmax(np.where(above_lcl, inter["increasing_x"], np.nan))          # PF:1129
    lfc_t = nanmax(np.where(inter["increasing_x"] == lfc_p[None, :],
                            inter["increasing_y"], np.nan))                     # PF:1131
    el_p = nanmin(above["decreasing_x"])                                        # PF:1136
    el_t = nanmax(np.where(inter["decreasing_x"] == el_p[None, :],
                           above["decreasing_y"], np.nan))                      # PF:1137

    temps_available = ~np.isnan(a) & ~np.isnan(b)                               # PF:1143
    top_p = nanmin(np.where(temps_available, pressure, np.nan))
    top_mask = pressure == top_p[None, :]                                       # PF:1145
    top_prof = nanmax(np.where(top_mask, a, np.nan))
    top_env = nanmax(np.where(top_mask, b, np.nan))
    if not np.array_equal(np.isnan(top_env), np.isnan(nanmax(b))):              # PF:1149
        raise ReferenceAssertion("Top temperature is NaN.")
    with np.errstate(invalid="ignore"):
        top_colder = top_prof <= top_env                                        # PF:1151
        el_exists = top_colder & (el_p < lcl_p)                                 # PF:1152-1153
    el_p = np.where(el_exists, el_p, np.nan)
    el_t = np.where(el_exists, el_t, np.nan)

    lfc_missing = np.isnan(nanmax(inter["increasing_x"]))                       # PF:1161
    with np.errstate(invalid="ignore"):
        lev_above = pressure < lcl_p[None, :]                                   # PF:1166
        pos_parcel = (np.where(lev_above, a, np.nan) > np.where(lev_above, b, np.nan)).any(axis=0)
        no_lfc_pos_parcel = pos_parcel & lfc_missing                            # PF:1170
        exists_but_na = ~lfc_missing & np.isnan(lfc_p)                          # PF:1174
        lfc_below_el_above = exists_but_na & (el_p < lcl_p)                     # PF:1176-1177
    replace = no_lfc_pos_parcel | lfc_below_el_above                            # PF:1180
    lfc_p = np.where(replace, lcl_p, lfc_p)
    lfc_t = np.where(replace, lcl_t, lfc_t)
    return {"lfc_pressure": lfc_p, "lfc_temperature": lfc_t,
            "el_pressure": el_p, "el_temperature": el_t}


# --------------------------------------------------------------------------- PF:164-206
def trapz(dat, x, mask=None, only_positive=False, only_negative=False):
    """PF:164-206.  ``dat``: dict of [M,N] containing key ``x``; ``mask`` [M,N] bool labelled by
    lower level.  Returns dict of [N] (one integral per variable)."""
    assert not (only_positive and only_negative)
    xv = dat[x]
    M = xv.shape[0]
    with np.errstate(all="ignore"):
        dx = np.abs(np.diff(xv, axis=0))                                        # PF:186, relabelled -1
        out = {}
        for k, v in dat.items():
            means = (v[:-1] + v[1:]) / 2                                        # PF:188 rolling(2).mean
            d = dx
            if mask is not None:
                d = np.where(mask[:M - 1], dx, np.nan)                          # PF:195
                means = np.where(mask[:M - 1], means, np.nan)
            areas = d * means
            if only_positive:
                areas = np.where(areas > 0, areas, np.nan)
            if only_negative:
                areas = np.where(areas < 0, areas, np.nan)
            out[k] = nansum(areas)
    return out


# --------------------------------------------------------------------------- PF:1200-1289
def trap_around_zeros(x, y, log_x=True):
    """PF:1200-1289 with start=0.  Returns (areas dict of [2M-1,N], mask [M,N])."""
    M, N = x.shape
    zi = find_intersections(x, y, np.zeros_like(y), log_x=log_x)                # PF:1225
    zero_y = zi["all_intersect_y"]                                              # labels 1..M-1
    zero_x = zi["all_intersect_x"]
    with np.errstate(all="ignore"):
        if log_x:
            x = np.log(x)
            zero_x = np.log(zero_x)
        after_mask = ~np.isnan(zero_y)                                          # labels 1..M-1
        before_mask = np.zeros((M, N), dtype=bool)                              # labels 0..M-1
        before_mask[:M - 1] = ~np.isnan(zero_y)                                 # PF:1242-1244

        # areas before zeros (shift_x=1), labels 0..M-1                           PF:1272
        xb = np.where(before_mask, x, np.nan)
        yb = np.where(before_mask, y, np.nan)
        dxb = np.full((M, N), np.nan)
        dxb[:M - 1] = xb[:M - 1] - zero_x                                       # PF:1258-1259
        bef = {"area": (yb / 2) * np.abs(dxb), "x": xb - dxb / 2, "dx": np.abs(dxb)}
        # areas after zeros (shift_x=0), labels 1..M-1                            PF:1273
        xa = np.where(after_mask, x[1:], np.nan)
        ya = np.where(after_mask, y[1:], np.nan)
        dxa = xa - zero_x
        aft = {"area": (ya / 2) * np.abs(dxa), "x": xa - dxa / 2, "dx": np.abs(dxa)}
        areas = {k: np.concatenate([bef[k], aft[k]], axis=0) for k in bef}      # PF:1276
        areas["x_from"] = areas["x"] - areas["dx"] / 2
        areas["x_to"] = areas["x"] + areas["dx"] / 2
    mask = np.isnan(bef["area"])                                                # PF:1285-1287
    return areas, mask


# --------------------------------------------------------------------------- PF:1291-1392
def cape_cin_base(pressure, temperature, lfc_pressure, el_pressure, parcel_temperature,
                  pos_cape_neg_cin=True, post_zero_cin=False):
    """PF:1291-1392.  Returns dict(cape, cin) [N]."""
    pressure = _as2d(pressure)
    M, N = pressure.shape
    b = _as2d(temperature, N)
    a = _as2d(parcel_temperature, N)
    lfc_p = np.broadcast_to(np.asarray(lfc_pressure, dtype=np.float64), (N,))
    el_p = np.broadcast_to(np.asarray(el_pressure, dtype=np.float64), (N,))
    el_p = np.where(np.isnan(el_p), nanmin(pressure), el_p)                     # PF:1329
    with np.errstate(all="ignore"):
        temp_diffs = {"temp_diff": a - b, "pressure": pressure,
                      "log_pressure": np.log(pressure)}                         # PF:1334
        areas, trapz_mask = trap_around_zeros(pressure, temp_diffs["temp_diff"], log_x=True)
        ax = np.exp(areas["x"])                                                 # PF:1347

        in_cape = (pressure <= lfc_p[None, :]) & (pressure >= el_p[None, :])    # PF:1352-1353
        d_cape = {k: np.where(in_cape, v, np.nan) for k, v in temp_diffs.items()}
        a_cape = np.where((ax <= lfc_p[None, :]) & (ax >= el_p[None, :]), areas["area"], np.nan)
        if pos_cape_neg_cin:
            a_cape = np.where(a_cape > 0, a_cape, np.nan)                       # PF:1359
        cape = th.RD * trapz(d_cape, "log_pressure", mask=trapz_mask,
                             only_positive=pos_cape_neg_cin)["temp_diff"]       # PF:1361
        cape = cape + th.RD * nansum(a_cape)                                    # PF:1365

        in_cin = pressure >= lfc_p[None, :]                                     # PF:1371
        d_cin = {k: np.where(in_cin, v, np.nan) for k, v in temp_diffs.items()}
        a_cin = np.where(ax >= lfc_p[None, :], areas["area"], np.nan)           # PF:1372
        if pos_cape_neg_cin:
            a_cin = np.where(a_cin < 0, a_cin, np.nan)                          # PF:1376
        cin = th.RD * trapz(d_cin, "log_pressure", mask=trapz_mask,
                            only_negative=pos_cape_neg_cin)["temp_diff"]        # PF:1378
        cin = cin + th.RD * nansum(a_cin)                                       # PF:1382
        if post_zero_cin:
            cin = np.where(cin <= 0, cin, 0.0)                                  # PF:1388
    return {"cape": cape, "cin": cin}


# --------------------------------------------------------------------------- PF:1394-1514
def cape_cin(pressure, temperature, dewpoint, parcel_temperature, parcel_pressure,
             parcel_dewpoint, opts, virtual_temperature_correction=True, lcl_interp="log",
             **kwargs):
    """PF:1394-1475.  Returns (dict(cape, cin), profile dict incl. lfc/el)."""
    profile = parcel_profile_with_lcl(pressure, temperature, dewpoint, parcel_pressure,
                                      parcel_temperature, parcel_dewpoint, opts,
                                      lcl_interp=lcl_interp)
    if not virtual_temperature_correction:
        pt, et, lt = "temperature", "environment_temperature", "lcl_temperature"
    else:
        pt, et, lt = ("virtual_temperature", "environment_virtual_temperature",
                      "lcl_virtual_temperature")
    le = lfc_el(profile["pressure"], profile[pt], profile[et],
                profile["lcl_pressure"], profile[lt])
    cc = cape_cin_base(profile["pressure"], profile[et], le["lfc_pressure"],
                       le["el_pressure"], profile[pt], **kwargs)
    profile = dict(profile)
    profile.update(le)
    return cc, profile


def surface_based_cape_cin(pressure, temperature, dewpoint, opts, **kwargs):
    """PF:1477-1514."""
    pressure = _as2d(pressure)
    N = pressure.shape[1]
    temperature = _as2d(temperature, N)
    dewpoint = _as2d(dewpoint, N)
    return cape_cin(pressure, temperature, dewpoint, parcel_temperature=temperature[0],
                    parcel_pressure=pressure[0], parcel_dewpoint=dewpoint[0], opts=opts,
                    **kwargs)


# --------------------------------------------------------------------------- PF:63-289
def bound_pressure(pressure, bound):
    """PF:208-227: closest level pressure to ``bound``; ties -> larger pressure."""
    with np.errstate(invalid="ignore"):
        diffs = np.abs(pressure - bound[None, :])
        return nanmax(np.where(diffs == nanmin(diffs)[None, :], pressure, np.nan))


def get_layer(dat, depth=100, interpolate=True):
    """PF:63-100.  ``dat`` dict of [L,N] containing 'pressure'."""
    bottom = nanmax(dat["pressure"])                                            # PF:80
    if interpolate:
        top = bottom - depth
        interp_level = log_interp(dat, dat["pressure"], top)                    # PF:85
        interp_level["pressure"] = top
        dat = insert_level(dat, interp_level, "pressure")                       # PF:89
    else:
        top = bound_pressure(dat["pressure"], bottom - depth)                   # PF:92
    p = dat["pressure"]
    with np.errstate(invalid="ignore"):
        keep = (p <= bottom[None, :]) & (p >= top[None, :])                     # PF:97-98
    # dat.where(cond) masks every variable, pressure included
    return {k: np.where(keep, v, np.nan) for k, v in dat.items()}


def most_unstable_parcel(dat, depth=300):
    """PF:102-135.  Returns dict(pressure, temperature, dewpoint) [N]."""
    layer = get_layer(dat, depth=depth, interpolate=False)
    eq = th.equivalent_potential_temperature(layer["pressure"], layer["temperature"],
                                             layer["dewpoint"])                 # PF:123
    max_eq = nanmax(eq)
    pres = nanmax(np.where(eq == max_eq[None, :], layer["pressure"], np.nan))   # PF:128
    is_mu = layer["pressure"] == pres[None, :]
    counts = np.where(~np.isnan(pres), is_mu.sum(axis=0), np.nan)               # PF:130
    if np.any(~np.isnan(counts)):
        if not (np.nanmax(counts) == np.nanmin(counts) == 1):                   # PF:131
            raise ReferenceAssertion("Vertical pressures are not unique")
    return {k: nanmax(np.where(is_mu, v, np.nan)) for k, v in layer.items()}    # PF:133


def mixed_layer(dat, depth=100):
    """PF:137-162."""
    layer = get_layer(dat, depth=depth)
    pressure_depth = np.abs(nanmin(layer["pressure"]) - nanmax(layer["pressure"]))
    tz = trapz(layer, "pressure")
    with np.errstate(all="ignore"):
        return {k: (1. / pressure_depth) * v for k, v in tz.items()}


def mixed_parcel(pressure, temperature, dewpoint, depth=100):
    """PF:229-289.  dict(theta, mixing_ratio, temperature, vapour_pressure, dewpoint, pressure)."""
    pressure = _as2d(pressure)
    N = pressure.shape[1]
    temperature = _as2d(temperature, N)
    dewpoint = _as2d(dewpoint, N)
    parcel_start_pressure = pressure[0]                                         # PF:250
    theta = th.potential_temperature(pressure, temperature)                     # PF:253
    mr = th.saturation_mixing_ratio(pressure, dewpoint)                         # PF:258
    mp = mixed_layer({"pressure": pressure, "theta": theta, "mixing_ratio": mr}, depth=depth)
    mp["temperature"] = mp["theta"] * th.exner_function(parcel_start_pressure)  # PF:268
    mp["vapour_pressure"] = th.vapor_pressure(parcel_start_pressure, mp["mixing_ratio"])
    mp["dewpoint"] = th.dewpoint_from_vapor_pressure(mp["vapour_pressure"])     # PF:280-282
    mp["pressure"] = parcel_start_pressure                                      # PF:287
    return mp


# --------------------------------------------------------------------------- PF:1517-1720
def shift_out_nans(x, name):
    """PF:1699-1720: per column, shift down until level 0 of ``name`` is not NaN."""
    x = {k: v.copy() for k, v in x.items()}
    L = x[name].shape[0]
    for _ in range(L):
        lead = np.isnan(x[name][0])
        if not lead.any():
            break
        for k in x:
            shifted = np.concatenate([x[k][1:], np.full((1,) + x[k].shape[1:], np.nan)], axis=0)
            x[k] = np.where(lead[None, :], shifted, x[k])
    return x


def dropna_all(dat):
    """Dataset.dropna(dim=vert_dim, how='all') (PF:1552, PF:1637): drop a level only if every
    variable is NaN in every column there."""
    alive = np.zeros(next(iter(dat.values())).shape[0], dtype=bool)
    for v in dat.values():
        alive |= (~np.isnan(v)).any(axis=1)
    return {k: v[alive] for k, v in dat.items()}, alive


def from_most_unstable_parcel(pressure, temperature, dewpoint, depth=300):
    """PF:1517-1555."""
    dat = {"pressure": pressure, "temperature": temperature, "dewpoint": dewpoint}
    unstable_layer = most_unstable_parcel(dat, depth=depth)
    with np.errstate(invalid="ignore"):
        keep = pressure <= unstable_layer["pressure"][None, :]                  # PF:1551
    dat = {k: np.where(keep, v, np.nan) for k, v in dat.items()}
    dat, _ = dropna_all(dat)                                                    # PF:1552
    dat = shift_out_nans(dat, "pressure")                                       # PF:1553
    return dat["pressure"], dat["temperature"], dat["dewpoint"], unstable_layer


def most_unstable_cape_cin(pressure, temperature, dewpoint, opts, depth=300, **kwargs):
    """PF:1557-1602.  Returns (cape_cin, profile, unstable_layer)."""
    pressure = _as2d(pressure)
    N = pressure.shape[1]
    temperature = _as2d(temperature, N)
    dewpoint = _as2d(dewpoint, N)
    p, t, td, ul = from_most_unstable_parcel(pressure, temperature, dewpoint, depth=depth)
    if p.shape[0] == 0:     # every level dropped (all-NaN input): keep one NaN level
        p = t = td = np.full((1, N), np.nan)
    res, profile = cape_cin(p, t, td, parcel_temperature=ul["temperature"],
                            parcel_pressure=ul["pressure"], parcel_dewpoint=ul["dewpoint"],
                            opts=opts, **kwargs)
    return res, profile, ul


def mix_layer(pressure, temperature, dewpoint, depth=100):
    """PF:1604-1649."""
    mp = mixed_parcel(pressure, temperature, dewpoint, depth=depth)
    with np.errstate(invalid="ignore"):
        keep = pressure < (nanmax(pressure) - depth)[None, :]                   # PF:1636
    dat = {"pressure": np.where(keep, pressure, np.nan),
           "temperature": np.where(keep, temperature, np.nan),
           "dewpoint": np.where(keep, dewpoint, np.nan)}
    dat, _ = dropna_all(dat)                                                    # PF:1637
    dat = shift_out_nans(dat, "pressure")                                       # PF:1638
    p = np.concatenate([mp["pressure"][None, :], dat["pressure"]], axis=0)      # PF:1642-1644
    t = np.concatenate([mp["temperature"][None, :], dat["temperature"]], axis=0)
    td = np.concatenate([mp["dewpoint"][None, :], dat["dewpoint"]], axis=0)
    return p, t, td, mp


def mixed_layer_cape_cin(pressure, temperature, dewpoint, opts, depth=100, **kwargs):
    """PF:1651-1697.  Returns (cape_cin, profile, mixed parcel)."""
    pressure = _as2d(pressure)
    N = pressure.shape[1]
    temperature = _as2d(temperature, N)
    dewpoint = _as2d(dewpoint, N)
    p, t, td, mp = mix_layer(pressure, temperature, dewpoint, depth=depth)
    res, profile = cape_cin(p, t, td, parcel_temperature=mp["temperature"],
                            parcel_pressure=mp["pressure"], parcel_dewpoint=mp["dewpoint"],
                            opts=opts, **kwargs)
    return res, profile, mp


# --------------------------------------------------------------------------- PF:1722-1756
def lifted_index(profile):
    """PF:1722-1756: environment minus parcel temperature, log-interpolated to 500 hPa."""
    N = profile["pressure"].shape[1]
    sel = {k: profile[k] for k in ("temperature", "environment_temperature")}
    dat = log_interp(sel, profile["pressure"], np.full(N, 500.0))
    return dat["environment_temperature"] - dat["temperature"]


# --------------------------------------------------------------------------- PF:1830-2259
def isobar_temperature(pressure, temperature, isobar):
    """PF:2193-2214."""
    N = pressure.shape[1]
    return log_interp({"t": temperature}, pressure, np.full(N, float(isobar)))["t"]


def deep_convective_index(pressure, temperature, dewpoint, lifted_index_):
    """PF:1830-1870."""
    N = pressure.shape[1]
    dat = log_interp({"temperature": temperature, "dewpoint": dewpoint}, pressure, np.full(N, 850.0))
    return (dat["temperature"] - 273.15) + (dat["dewpoint"] - 273.15) - lifted_index_


def lapse_rate(pressure, temperature, height, from_pressure=700, to_pressure=500):
    """PF:2102-2135."""
    N = pressure.shape[1]
    lo = log_interp({"t": temperature, "h": height}, pressure, np.full(N, float(from_pressure)))
    hi = log_interp({"t": temperature, "h": height}, pressure, np.full(N, float(to_pressure)))
    with np.errstate(all="ignore"):
        return (hi["t"] - lo["t"]) / (hi["h"] / 1000 - lo["h"] / 1000)


def freezing_level_height(temperature, height, level=273.15):
    """PF:2137-2160."""
    inter = find_intersections(height, temperature, np.full_like(temperature, level))
    return nanmin(inter["all_intersect_x"])


def wet_bulb_temperature_fast(temperature, dewpoint):
    """PF:364-387."""
    return temperature - (1 / 3) * (temperature - dewpoint)


def wet_bulb_temperature(pressure, temperature, dewpoint, opts):
    """PF:389-445 (Normand's rule): lcl of every point, then moist_lapse from the LCL back to the point's
    pressure.  The reference loops over levels and calls moist_lapse on one level at a time; per point that
    is ``opts.moist_lapse(p, lcl_t, lcl_p)`` with a one-level profile."""
    shp = np.shape(temperature)
    p = np.broadcast_to(np.asarray(pressure, dtype=np.float64), shp).ravel()
    t = np.asarray(temperature, dtype=np.float64).ravel()
    td = np.asarray(dewpoint, dtype=np.float64).ravel()
    out = np.full(p.shape, np.nan)
    ok = ~(np.isnan(p) | np.isnan(t) | np.isnan(td))
    if ok.any():
        l = lcl(p[ok], t[ok], td[ok], opts)
        out[ok] = opts.moist_lapse(p[ok][None, :], l["lcl_temperature"], l["lcl_pressure"])[0]
    return out.reshape(shp)


def significant_hail_parameter(mucape, mixing_ratio, lapse, temp_500, shear, flh):
    """PF:2261-2306, xarray ``.where(cond, other)`` semantics (a failed comparison, also with NaN, takes
    ``other``; without ``other`` it gives NaN)."""
    with np.errstate(invalid="ignore"):
        mixing_ratio = mixing_ratio * 1e3
        lapse = -lapse
        temp_500 = temp_500 - 273.15
        shear = where(shear >= 7, shear)
        shear = where(shear <= 27, shear)
        mixing_ratio = where(mixing_ratio >= 11, mixing_ratio)
        mixing_ratio = where(mixing_ratio <= 13.6, mixing_ratio)
        temp_500 = where(temp_500 <= -5.5, temp_500, -5.5)
        ship = mucape * mixing_ratio * lapse * -temp_500 * shear / 42000000
        ship = where(mucape >= 1300, ship, ship * (mucape / 1300))
        ship = where(lapse >= 5.8, ship, ship * (lapse / 5.8))
        ship = where(flh >= 2400, ship, ship * (flh / 2400))
    return ship


def storm_proxies(dat):
    """PF:2323-2407 on a dict of [N] arrays as conv_properties returns them."""
    with np.errstate(invalid="ignore"):
        s06 = dat["shear_magnitude"]
        ml100 = where(dat["mixed_100_cape"] >= 0, dat["mixed_100_cape"])
        ml50 = where(dat["mixed_50_cape"] >= 0, dat["mixed_50_cape"])
        mu = where(dat["mu_cape"] >= 0, dat["mu_cape"])
        out = {}
        out["proxy_Craven2004"] = (ml100 * s06) >= 20000
        out["proxy_Kunz2007"] = np.logical_or(dat["mixed_100_lifted_index"] <= -2.07,
                                              np.logical_or(mu >= 1474, dat["mixed_100_dci"] >= 25.7))
        tr = np.logical_and(ml100 * s06 >= 10000, ml100 >= 100)
        tr = np.logical_and(tr, s06 >= 5)
        out["proxy_Trapp2007"] = np.logical_and(tr, dat["positive_shear"])
        out["proxy_Marsh2009"] = (ml100 * s06) >= 10000
        out["proxy_Allen2011"] = ml50 * s06 ** 1.67 >= 25000
        al = np.logical_and(out["proxy_Allen2011"], dat["mixed_50_cin"] > -25)
        al = np.logical_and(al, s06 > 7.5)
        out["proxy_Allen2014"] = np.logical_and(al, dat["lapse_rate_700_500"] < -6.5)
        out["proxy_Eccel2012"] = np.logical_and(ml100 * s06 > 10000, dat["mixed_100_cin"] > -50)
        mo = np.logical_or(dat["mixed_100_lifted_index"] <= -1.6, ml100 >= 439)
        out["proxy_Mohr2013"] = np.logical_or(mo, dat["mixed_100_dci"] >= 26.4)
        out["ship"] = significant_hail_parameter(mu, dat["mu_mixing_ratio"], dat["lapse_rate_700_500"],
                                                 dat["temp_500"], s06, dat["freezing_level"])
        out["proxy_SHIP_0.1"] = out["ship"] > 0.1
    return out


def wind_shear(surface_wind_u, surface_wind_v, wind_u, wind_v, height, shear_height=6000):
    """PF:2216-2259."""
    N = wind_u.shape[1]
    hi = linear_interp({"u": wind_u, "v": wind_v}, height, np.full(N, float(shear_height)))
    su, sv = hi["u"] - surface_wind_u, hi["v"] - surface_wind_v
    with np.errstate(invalid="ignore"):
        return {"shear_u": su, "shear_v": sv, "shear_magnitude": np.sqrt(su ** 2 + sv ** 2),
                "positive_shear": np.sqrt(hi["u"] ** 2 + hi["v"] ** 2) > np.sqrt(surface_wind_u ** 2 + surface_wind_v ** 2)}


def conv_properties(dat, opts, min_set=False, ignore_nans=False):
    """PF:1951-2100 (min_set: PF:1872-1949 min_conv_properties).  ``dat``: dict of [L,N] arrays pressure,
    temperature, specific_humidity, height_asl, wind_u, wind_v, wind_height_above_surface and [N] arrays
    surface_wind_u, surface_wind_v.  ``ignore_nans`` skips the mask of columns with a NaN input (PF:1976-1983),
    which min_set never applies.  Returns a flat dict of [N] arrays."""
    p, t = dat["pressure"], dat["temperature"]
    td = th.dewpoint_from_specific_humidity(p, t, dat["specific_humidity"], opts.metpy_compat)
    out = {}

    def add_parcel(prefix, cc, prof):
        out[prefix + "_cape"], out[prefix + "_cin"] = cc["cape"], cc["cin"]
        li = lifted_index(prof)
        out[prefix + "_lifted_index"] = li
        out[prefix + "_dci"] = deep_convective_index(p, t, td, li)

    cc, prof, _ = mixed_layer_cape_cin(p, t, td, opts, depth=100)
    if min_set:
        out["mixed_100_cape"], out["mixed_100_cin"] = cc["cape"], cc["cin"]
        out["mixed_100_lifted_index"] = lifted_index(prof)
    else:
        add_parcel("mixed_100", cc, prof)
        cc, prof, mu_parcel = most_unstable_cape_cin(p, t, td, opts, depth=250)
        add_parcel("mu", cc, prof)
        cc, prof, _ = mixed_layer_cape_cin(p, t, td, opts, depth=50)
        add_parcel("mixed_50", cc, prof)
        out["mu_mixing_ratio"] = th.saturation_mixing_ratio(mu_parcel["pressure"], mu_parcel["dewpoint"])
    out["lapse_rate_700_500"] = lapse_rate(p, t, dat["height_asl"])
    out["temp_500"] = isobar_temperature(p, t, 500)
    out["freezing_level"] = freezing_level_height(t, dat["height_asl"])
    out["melting_level"] = freezing_level_height(wet_bulb_temperature_fast(t, td), dat["height_asl"])
    out.update(wind_shear(dat["surface_wind_u"], dat["surface_wind_v"], dat["wind_u"], dat["wind_v"],
                          dat["wind_height_above_surface"], 6000))
    if not min_set and not ignore_nans:
        valid = ~(np.isnan(td).any(0) | np.isnan(p).any(0) | np.isnan(t).any(0) |
                  np.isnan(dat["specific_humidity"]).any(0))                      # PF:1976-1983, 2098-2099
        out = {k: np.where(valid, v, np.nan) for k, v in out.items()}
    return out


# --------------------------------------------------------------------------- suite
def suite(pressure, temperature, dewpoint, opts, ml_depth=100, mu_depth=300, **kwargs):
    """The SB + ML + MU suite the benchmark metric is quoted on (the hot-path part of
    parcel_test.py:416-547 ``conv_properties_xarray``).  Returns a flat dict of [N] arrays."""
    out = {}
    sb, sbp = surface_based_cape_cin(pressure, temperature, dewpoint, opts, **kwargs)
    ml, mlp, mp = mixed_layer_cape_cin(pressure, temperature, dewpoint, opts, depth=ml_depth,
                                       **kwargs)
    mu, mup, ul = most_unstable_cape_cin(pressure, temperature, dewpoint, opts, depth=mu_depth,
                                         **kwargs)
    for pre, cc, prof in (("sb", sb, sbp), ("ml", ml, mlp), ("mu", mu, mup)):
        out[pre + "_cape"] = cc["cape"]
        out[pre + "_cin"] = cc["cin"]
        for k in ("lcl_pressure", "lcl_temperature", "lcl_virtual_temperature", "lfc_pressure",
                  "lfc_temperature", "el_pressure", "el_temperature"):
            out[pre + "_" + k] = prof[k]
    for k in ("pressure", "temperature", "dewpoint"):
        out["ml_parcel_" + k] = mp[k]
        out["mu_parcel_" + k] = ul[k]
    return out
