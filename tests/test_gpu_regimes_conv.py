"""conv_properties / min_conv_properties and storm_proxies on the real-world regimes of tests/regime_columns.py against
the float64 oracle's assembly of the same steps (oracle.parcel.conv_properties and storm_proxies).

The chain behind conv_properties is about a dozen GPU calls: q -> Td, three parcel lifts with profile rows, the
interpolations of the lifted index, DCI, T500 and the 700-500 hPa lapse rate, the freezing and melting level crossings,
the 0-6 km shear, the MU mixing ratio and the NaN mask, then storm_proxies.  The regimes take it where these kernels
branch: high terrain leaves 850 / 700 hPa unbracketed (no extrapolation: NaN), cold columns have no 0 C crossing, ERA5
extrapolation puts crossings below ground, the ERA5 levels hit 850 / 700 / 500 hPa exactly, masked below-ground levels
put NaN fields at a bracketing coordinate, and some columns carry q = 0 or q < 0 on their top levels (NaN dewpoints).

Every case runs in float64 NumPy, float32 NumPy and float32 CUDA tensors; on the shared ERA5 axis also with the same
pressures as a contiguous [L, N] array.  NaN patterns must equal the oracle's in every output.  Values are held to
bounds derived below from the rounding of the inputs and the documented error of each upstream output; the exact
(float64) route to rtol = atol = 1e-8, the bound test_gpu_derived.test_conv_properties_assembly holds.  Layouts and
array types must not change a bit, and a shared 1-D pressure axis must broadcast along the vertical axis whatever the
number of columns.
"""

import numpy as np
import pytest
import torch

import regime_columns as rc
from oracle import parcel as op
from oracle import tables as otab
from oracle import thermo as th
from test_gpu_parity import FAST_BOUND
from xarray_parcel_b200 import _lib
import xarray_parcel_b200.parcel_functions as parcel

pytestmark = pytest.mark.gpu

N_COLUMNS = 2000
# id: (regime, regime_columns.columns keywords).  70 model levels (per-column pressure), the 0.01 hPa top at 137 levels
# (every column handed over to the float64 fix-up, as on above_1100), and the 37 ERA5 levels as a shared 1-D axis.
CASES = {
    "terrain": ("terrain", {}),
    "cold": ("cold", {}),
    "moist_heat": ("moist_heat", {}),
    "high_surface": ("high_surface", {}),
    "above_1100": ("above_1100", {}),
    "top0.01_L137": ("synth_like", dict(levels=137, p_top=0.01)),
    "cold_era5": ("cold", dict(layout="era5")),
    "moist_heat_era5": ("moist_heat", dict(layout="era5")),
    "terrain_era5": ("terrain", dict(layout="era5")),
    "masked_era5": ("masked", dict(layout="era5_masked")),
}
AXIS_CASES = [c for c, (_, kw) in CASES.items() if kw.get("layout", "model") != "model"]
ALL_HANDED_OVER = ("above_1100", "top0.01_L137")
# how the call is made: (dtype, torch CUDA tensors, shared axis passed as a contiguous [L, N] array)
VARIANTS = {"f64": (np.float64, False, False), "f32": (np.float32, False, False),
            "f32-cuda": (np.float32, True, False), "f64-pcol": (np.float64, False, True),
            "f32-pcol": (np.float32, False, True)}
PARAMS = [(c, v, False) for c in CASES for v in VARIANTS if not v.endswith("pcol") or c in AXIS_CASES]
PARAMS += [("masked_era5", v, True) for v in VARIANTS]

# ---- bounds ----------------------------------------------------------------------------------------------------------
# U: float32 unit roundoff; one rounding of x moves it by at most U * |x|.  ULP300: the float32 ulp on [256, 512) K.
U = 2.0 ** -24
ULP300 = 2.0 ** -15
# The kernels evaluate in float64 in another operation order than NumPy: a relative difference far below 1e-12.
F64_NOISE = 1e-12
# Second-order terms of the first-order propagations below are O(U^2) relative: a factor 1.01 covers them.
SECOND_ORDER = 1.01
# The exact (float64) route: the bound of test_gpu_derived.test_conv_properties_assembly.
EXACT_RTOL = EXACT_ATOL = 1e-8
# The fast routes' parcel_profile_with_lcl rows (every row, pressure included) and ML / MU parcels against the oracle:
# the bounds test_gpu_regimes holds them to.
PROFILE_RTOL = 3e-6
PARCEL_RTOL = 3e-7
# Steepest temperature profile in ln p [K]: a dry adiabat kappa * T (86 K at 300 K); the regimes' environmental lapse
# rates (<= 9.5 K/km, 6.5 below ground) give Rd / g * lapse * T < 85 K at 300 K.
SLOPE_MAX = 100.0
# Columns allowed near a threshold (flags) or with a wet-bulb temperature within its rounding of 273.15 K.
NEAR_CAP = 0.005

PARCELS = ("mu", "mixed_100", "mixed_50")


# ---- fixtures ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    c = _lib.get_context(0)
    if not c.tables_loaded():
        c.tables_build()
    return c


@pytest.fixture(scope="module")
def gpu_tables(ctx):
    idx, cur = ctx.tables_get()
    pl, tl = otab.default_grids()
    return otab.AdiabatTables(pl, tl, idx, cur)


def _compat(case):
    return "1.4.1" if list(CASES).index(case) % 2 == 0 else "1.6.2"


class _Cache:
    """Inputs, oracle results and GPU results per case, computed once for the module."""

    def __init__(self, tables):
        self.tables, self.store = tables, {}

    def get(self, key, make):
        if key not in self.store:
            self.store[key] = make()
        return self.store[key]

    def fields(self, case):
        """float32 conv_properties inputs of a case (pressure [37] on the ERA5 layouts, [L, N] otherwise)."""
        def make():
            regime, kw = CASES[case]
            i = list(CASES).index(case)
            p, t, td, p0 = rc.columns(regime, N_COLUMNS, seed=600 + i, **kw)
            return rc.conv_fields(p, t, td, p0, seed=700 + i)
        return self.get(("fields", case), make)

    def wide(self, case):
        """The float64-widened inputs with the pressure broadcast to [L, N], and the oracle's dewpoint."""
        def make():
            d = {k: v.astype(np.float64) for k, v in self.fields(case).items()}
            if d["pressure"].ndim == 1:
                d["pressure"] = np.ascontiguousarray(np.broadcast_to(d["pressure"][:, None], d["temperature"].shape))
            d["dewpoint"] = th.dewpoint_from_specific_humidity(d["pressure"], d["temperature"],
                                                              d["specific_humidity"], _compat(case))
            return d
        return self.get(("wide", case), make)

    def oracle(self, case, min_set, ignore_nans):
        def make():
            d = self.wide(case)
            opts = op.Options(op.MoistLapseLUT(self.tables), lcl_mode="converged", metpy_compat=_compat(case))
            dat = {k: v for k, v in d.items() if k != "dewpoint"}
            with np.errstate(all="ignore"):
                out = op.conv_properties(dat, opts, min_set=min_set, ignore_nans=ignore_nans)
                prox = op.storm_proxies(out) if not min_set else {}
            return out, prox
        return self.get(("oracle", case, min_set, ignore_nans), make)

    def aux(self, case):
        """Oracle intermediates the bounds read: T, height at 700 / 500 hPa, the wind at 6 km, the 1/3-rule wet bulb."""
        def make():
            d = self.wide(case)
            P, T, H, D = d["pressure"], d["temperature"], d["height_asl"], d["dewpoint"]
            n = T.shape[1]
            with np.errstate(all="ignore"):
                lo = op.log_interp({"t": T, "h": H}, P, np.full(n, 700.0))
                hi = op.log_interp({"t": T, "h": H}, P, np.full(n, 500.0))
                w = op.linear_interp({"u": d["wind_u"], "v": d["wind_v"]}, d["wind_height_above_surface"],
                                     np.full(n, 6000.0))
                wb = op.wet_bulb_temperature_fast(T, D)
                dwb = SECOND_ORDER * U * (np.abs(wb) + np.abs(D) / 3 + np.abs(T - D))
            return dict(t700=lo["t"], h700=lo["h"], t500=hi["t"], h500=hi["h"], hu=w["u"], hv=w["v"], wb=wb, dwb=dwb,
                        h=H, ws=np.hypot(w["u"], w["v"]), ss=np.hypot(d["surface_wind_u"], d["surface_wind_v"]))
        return self.get(("aux", case), make)


@pytest.fixture(scope="module")
def cache(gpu_tables):
    return _Cache(gpu_tables)


REPORT = {}


@pytest.fixture(scope="module", autouse=True)
def report():
    """Per (case, call): the largest |GPU - oracle| of every output and its ratio to the bound; printed at the end of
    the module (pytest -s)."""
    yield REPORT
    if REPORT:
        print("\ncase / call / output                                   max |err|   err/bound  near-excused")
        for k in sorted(REPORT):
            err, ratio, near = REPORT[k]
            print(f"{k:<54} {err:10.3g} {ratio:10.3g}  {near}")


# ---- calls -----------------------------------------------------------------------------------------------------------
def _inputs(cache, case, variant):
    dtype, cuda, pcol = VARIANTS[variant]
    d = {k: v.astype(dtype) for k, v in cache.fields(case).items()}
    if pcol:
        d["pressure"] = np.ascontiguousarray(np.broadcast_to(d["pressure"][:, None], d["temperature"].shape))
    if cuda:
        d = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in d.items()}
    return d


def _host(x):
    """A result (NumPy or torch, any dtype) as a NumPy array."""
    return x.cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def _f64(x):
    return _host(x).astype(np.float64)


def _run(cache, case, variant, ignore_nans, min_set):
    def make():
        dat = _inputs(cache, case, variant)
        if min_set:
            return dict(parcel.min_conv_properties(dict(dat), metpy_compat=_compat(case))), {}
        res = parcel.conv_properties(dict(dat), ignore_nans=ignore_nans, metpy_compat=_compat(case))
        return dict(res), dict(parcel.storm_proxies(res))
    return cache.get(("run", case, variant, ignore_nans, min_set), make)


def _route(ctx, cache, case, variant):
    """The lifting route conv_properties takes: most_unstable_cape_cin called with its arguments.  Returns
    (launches, last_exact_count, MU parcel dewpoint)."""
    dat = _inputs(cache, case, variant)
    n0 = ctx.launch_count()
    _, _, ul = parcel.most_unstable_cape_cin(dat["pressure"], dat["temperature"], dat["specific_humidity"], depth=250,
                                            metpy_compat=_compat(case), specific_humidity=True)
    return ctx.launch_count() - n0, ctx.last_exact_count(), _f64(ul["dewpoint"])


# ---- bounds per output ---------------------------------------------------------------------------------------------
def _bounds(o, aux, f32, mu_td):
    """Per-column bound of |GPU - oracle| for every float output of ``o`` (the oracle's conv_properties).

    float64 runs the exact kernel and the float64 interpolations: EXACT_RTOL / EXACT_ATOL everywhere.  float32:

    * CAPE / CIN: FAST_BOUND of test_gpu_parity (the fast routes; the exact kernel's float32 outputs are one rounding).
    * lifted index = T_env - T_parcel at 500 hPa, log-interpolated from the profile rows.  Each row value is within
      PROFILE_RTOL of the oracle's, and an interpolation is a convex combination, so the two interpolated temperatures
      move by at most PROFILE_RTOL * (|T_env| + |T_parcel|).  The LCL row's pressure is within PROFILE_RTOL too; as a
      bracketing coordinate it moves each interpolated temperature by at most SLOPE_MAX * PROFILE_RTOL (ln p moves by
      PROFILE_RTOL).  The two float32 interpolation outputs and the difference add 2 U * (|T_env| + |T_parcel|).
    * DCI = (T850 - 273.15) + (Td850 - 273.15) - LI in float32 tensor arithmetic: the LI bound, plus T850 (one rounding,
      1/2 ulp), Td850 (Td rounded once to float32, then the interpolation rounded: 1 ulp), 273.15 taken as a float32
      constant twice (0.2 ulp each) and three operations on results below 64 K (< 0.1 ulp at 300 K): under 2 ulps.
    * T500, freezing level: the float64 evaluation of float32 inputs rounded once: (U + F64_NOISE) * |x|.
    * melting level: the 1/3-rule wet bulb is evaluated in float32 (t - (1/3) * (t - td) with a rounded td):
      |dwb| <= U * (|wb| + |td| / 3 + |t - td|) per level (``aux["dwb"]``).  Moving both ends of the crossing segment by
      dwb moves the crossing height by dwb * |dh / dwb| over that segment (the two ends lie on opposite sides of
      273.15 K).  Columns with a level within dwb of 273.15 K may gain or lose a crossing: they are excused
      (``melting_near``), counted and capped.
    * lapse rate = (T500 - T700) / (h500 / 1000 - h700 / 1000) in float32 from four rounded interpolations: numerator
      off by U * (|T500| + |T700|) + U * |num|, denominator by 2 U * (|h500| + |h700|) / 1000 + U * |den| (the division
      by 1000 rounds too); propagated as (d_num + |lapse| * d_den) / |den| + U * |lapse|.  The numerator term is
      absolute: the 700-500 hPa difference may be near 0 in polar columns.
    * shear_u = hu - su with hu rounded once and su exact: U * |hu| + U * |shear_u|; magnitude: d_u + d_v plus 2 U for
      the squares, the sum and the square root.
    * MU mixing ratio w = eps e(Td) / (p - e(Td)) of the MU parcel (p and Td within PARCEL_RTOL):
      d ln w = p / (p - e) * (d ln p + 17.67 * 243.5 / (Td - 29.65)^2 * dTd), p / (p - e) = 1 + w / eps, plus the
      output rounding.  Td is the GPU parcel's (within PARCEL_RTOL of the oracle's: a negligible change of the factor).
    """
    B = {}
    keys = [k for k, v in o.items() if v.dtype != bool and k != "positive_shear"]
    if not f32:
        with np.errstate(invalid="ignore"):
            for k in keys:
                B[k] = EXACT_RTOL * np.abs(o[k]) + EXACT_ATOL
            B["melting_near"] = np.zeros(o["mixed_100_cape"].shape, dtype=bool)
        return B
    with np.errstate(invalid="ignore", divide="ignore"):
        te = np.abs(np.where(np.isnan(aux["t500"]), 330.0, aux["t500"]))
        for pre in PARCELS:
            if pre + "_cape" not in o:
                continue
            for f in ("cape", "cin"):
                rel, ab = FAST_BOUND[f]
                B[f"{pre}_{f}"] = rel * np.abs(o[f"{pre}_{f}"]) + ab
            temps = te + np.abs(te - np.nan_to_num(o[pre + "_lifted_index"]))
            B[pre + "_lifted_index"] = (PROFILE_RTOL + 2 * U) * temps + 2 * SLOPE_MAX * PROFILE_RTOL
            if pre + "_dci" in o:
                B[pre + "_dci"] = B[pre + "_lifted_index"] + 2 * ULP300
        for k in ("temp_500", "freezing_level"):
            B[k] = (U + F64_NOISE) * np.abs(o[k])
        # melting level
        _, slope, dwb = _lowest_crossing(aux)
        B["melting_level"] = SECOND_ORDER * dwb * slope + (U + F64_NOISE) * np.abs(o["melting_level"])
        with np.errstate(invalid="ignore"):
            B["melting_near"] = (np.abs(aux["wb"] - 273.15) <= aux["dwb"]).any(axis=0)
        # lapse rate
        num = aux["t500"] - aux["t700"]
        den = aux["h500"] / 1000 - aux["h700"] / 1000
        d_num = U * (np.abs(aux["t500"]) + np.abs(aux["t700"])) + U * np.abs(num)
        d_den = 2 * U * (np.abs(aux["h500"]) + np.abs(aux["h700"])) / 1000 + U * np.abs(den)
        lapse = o["lapse_rate_700_500"]
        B["lapse_rate_700_500"] = SECOND_ORDER * (d_num + np.abs(lapse) * d_den) / np.abs(den) + U * np.abs(lapse)
        # shear
        du = U * np.abs(aux["hu"]) + U * np.abs(o["shear_u"])
        dv = U * np.abs(aux["hv"]) + U * np.abs(o["shear_v"])
        B["shear_u"], B["shear_v"] = SECOND_ORDER * du, SECOND_ORDER * dv
        B["shear_magnitude"] = SECOND_ORDER * (du + dv) + 2 * U * np.abs(o["shear_magnitude"])
        # MU mixing ratio
        if "mu_mixing_ratio" in o:
            w = np.abs(o["mu_mixing_ratio"])
            k_td = 17.67 * 243.5 / (mu_td - 29.65) ** 2 * np.abs(mu_td)
            B["mu_mixing_ratio"] = (SECOND_ORDER * (1 + w / th.EPSILON) * (1 + k_td) * PARCEL_RTOL + U) * w
    return B


def _lowest_crossing(aux):
    """Per column of the oracle's wet bulb: the slope |dh / dwb| of the segment that gives the lowest crossing of
    273.15 K and the larger wet-bulb rounding bound of its two ends (NaN without a crossing)."""
    h, d = aux["h"], aux["wb"] - 273.15
    s = np.sign(d)
    with np.errstate(invalid="ignore", divide="ignore"):
        cross = (s[:-1] != s[1:]) & ~np.isnan(s[:-1]) & ~np.isnan(s[1:])
        ix = (d[1:] * h[:-1] - d[:-1] * h[1:]) / (d[1:] - d[:-1])
        ix = np.where(cross & ~np.isnan(ix), ix, np.inf)
        k = np.argmin(ix, axis=0)
        c = np.arange(h.shape[1])
        has = np.isfinite(ix[k, c])
        slope = np.abs(h[k + 1, c] - h[k, c]) / np.abs(d[k + 1, c] - d[k, c])
        dwb = np.maximum(aux["dwb"][k, c], aux["dwb"][k + 1, c])
    return np.where(has, ix[k, c], np.nan), np.where(has, slope, np.nan), np.where(has, dwb, np.nan)


def _near(x, bx, thr):
    with np.errstate(invalid="ignore"):
        return np.abs(x - thr) <= bx


def _flag_excuses(o, B, prox_ora, tie, f32):
    """Per storm-proxy flag: the columns where some input the flag tests lies within its bound of the threshold, so
    that the flag may differ (``tie``: the columns where positive_shear may differ).  CAPE's own test against 0 (a
    negative CAPE is ignored) needs no excuse: a CAPE within its bound (< 0.1 J/kg) of 0 fails every threshold of
    every flag, as a product with the shear or alone, whether it is ignored or not.

    SHIP is continuous at its clipping thresholds (1300 J/kg, 5.8 K/km, -5.5 C, 2400 m) and NaN outside its shear (7-27
    m/s) and mixing-ratio (11-13.6 g/kg) windows: columns near a window edge are excused.  Its bound is the sum of its
    inputs' relative bounds, MU CAPE and lapse rate counted twice (they enter squared below 1300 J/kg and 5.8 K/km), the
    500 hPa temperature relative to its clipped value (clipping is 1-Lipschitz), plus the output rounding.  Where MU CAPE
    lies within its bound of 0, SHIP is at most (0.1 J/kg)^2 / 1300 * 13.6 g/kg * 10 K/km * 60 K * 27 m/s / 4.2e7 <
    1e-9, and NaN where the CAPE came out below 0: its NaN pattern is excused there and its value held to 1e-9.
    Returns ({flag: mask}, SHIP bound, SHIP NaN excuse)."""
    with np.errstate(invalid="ignore", divide="ignore"):
        s06, bs = o["shear_magnitude"], B["shear_magnitude"]
        m100, b100 = o["mixed_100_cape"], B["mixed_100_cape"]
        m50, b50 = o["mixed_50_cape"], B["mixed_50_cape"]
        mu, bmu = o["mu_cape"], B["mu_cape"]
        p100 = m100 * s06
        bp100 = np.abs(s06) * b100 + np.abs(m100) * bs + b100 * bs
        p50 = m50 * np.abs(s06) ** 1.67
        bp50 = SECOND_ORDER * (np.abs(s06) ** 1.67 * b50 + np.abs(m50) * 1.67 * np.abs(s06) ** 0.67 * bs)
        li, bli = o["mixed_100_lifted_index"], B["mixed_100_lifted_index"]
        dci, bdci = o["mixed_100_dci"], B["mixed_100_dci"]
        ex = {
            "proxy_Craven2004": _near(p100, bp100, 20000),
            "proxy_Kunz2007": _near(li, bli, -2.07) | _near(mu, bmu, 1474) | _near(dci, bdci, 25.7),
            "proxy_Trapp2007": _near(p100, bp100, 10000) | _near(m100, b100, 100) | _near(s06, bs, 5) | tie,
            "proxy_Marsh2009": _near(p100, bp100, 10000),
            "proxy_Allen2011": _near(p50, bp50, 25000),
        }
        ex["proxy_Allen2014"] = (ex["proxy_Allen2011"] | _near(o["mixed_50_cin"], B["mixed_50_cin"], -25) |
                                 _near(s06, bs, 7.5) | _near(o["lapse_rate_700_500"], B["lapse_rate_700_500"], -6.5))
        ex["proxy_Eccel2012"] = _near(p100, bp100, 10000) | _near(o["mixed_100_cin"], B["mixed_100_cin"], -50)
        ex["proxy_Mohr2013"] = _near(li, bli, -1.6) | _near(m100, b100, 439) | _near(dci, bdci, 26.4)
        mr, bmr = o["mu_mixing_ratio"], B["mu_mixing_ratio"]
        lapse, bl = o["lapse_rate_700_500"], B["lapse_rate_700_500"]
        t5, bt5 = np.minimum(o["temp_500"] - 273.15, -5.5), B["temp_500"]
        flh, bf = o["freezing_level"], B["freezing_level"]
        window = _near(mr, bmr, 0.011) | _near(mr, bmr, 0.0136) | _near(s06, bs, 7) | _near(s06, bs, 27)
        rel = (2 * bmu / np.abs(mu) + bmr / np.abs(mr) + 2 * bl / np.abs(lapse) + bt5 / np.abs(t5) +
               bs / np.abs(s06) + bf / np.abs(flh))
        ship = prox_ora["ship"]
        b_ship = SECOND_ORDER * np.abs(ship) * rel + (U if f32 else F64_NOISE) * np.abs(ship)
        zero_cape = _near(mu, bmu, 0)
        b_ship = np.where(zero_cape, 1e-9, b_ship)
        window |= np.isfinite(ship) & ~np.isfinite(b_ship)
        ex["ship"] = window
        ex["proxy_SHIP_0.1"] = window | _near(ship, b_ship, 0.1)
    return ex, b_ship, zero_cape & ~window


def _positive_shear_tie(aux, f32):
    """positive_shear = |wind at 6 km| > |surface wind|: the columns where the two magnitudes lie within their bounds
    of each other.  float32: the 6 km wind rounded once, then squares, sum and root (3 U); the surface wind is an exact
    input (2 U).  float64: EXACT_RTOL / EXACT_ATOL on each."""
    hs, ss = aux["ws"], aux["ss"]
    tie = SECOND_ORDER * (3 * U * hs + 2 * U * ss) if f32 else EXACT_RTOL * (hs + ss) + 2 * EXACT_ATOL
    return _near(hs, tie, ss)


def _check(case, call, got, ora, B, what):
    """NaN patterns identical and |got - ora| <= B for every float output; returns the number of excused columns."""
    n = next(iter(ora.values())).shape[0]
    for k, v in ora.items():
        if k == "positive_shear":
            continue
        assert k in B, f"{what}{k} has no bound"
        a = _f64(got[k])
        excuse = B.get(k + "_excuse", np.zeros(n, dtype=bool))
        nan_excuse = excuse | B.get(k + "_nan_excuse", np.zeros(n, dtype=bool))
        mis = np.flatnonzero((np.isnan(a) != np.isnan(v)) & ~nan_excuse)
        assert mis.size == 0, (f"{what}{k}: NaN pattern differs from the oracle in columns {mis[:8]} "
                               f"(got {a[mis[:4]]}, oracle {v[mis[:4]]})")
        ok = ~np.isnan(v) & ~np.isnan(a) & ~excuse
        err = np.where(ok, np.abs(np.where(ok, a, 0.0) - np.where(ok, v, 0.0)), 0.0)
        with np.errstate(invalid="ignore", divide="ignore"):
            over = np.flatnonzero(ok & ~(err <= B[k]))
            ratio = float(np.nanmax(np.where(ok & (B[k] > 0), err / B[k], 0.0))) if n else 0.0
        assert over.size == 0, (f"{what}{k}: {over.size} columns outside the bound, e.g. "
                                f"{[(int(i), float(a[i]), float(v[i]), float(B[k][i])) for i in over[:4]]}")
        REPORT[f"{case} / {call} / {k}"] = (float(err.max()) if n else 0.0, ratio, int(excuse.sum()))


# ---- the regimes against the oracle ----------------------------------------------------------------------------------
@pytest.mark.parametrize("param", PARAMS, ids=[f"{c}-{v}" + ("-ignore_nans" if i else "") for c, v, i in PARAMS])
def test_conv_properties_regimes_against_oracle(ctx, cache, param):
    case, variant, ignore_nans = param
    dtype, cuda, pcol = VARIANTS[variant]
    f32 = dtype == np.float32
    n = N_COLUMNS
    shared = case in AXIS_CASES and not pcol
    # the route: float64 and the shared axis (profile rows are not on the shared-axis sweeps) take the exact kernel,
    # one launch; float32 per-column pressure the gather route with profile rows, two launches (sweep and fix-up)
    launches, n_exact, mu_td = _route(ctx, cache, case, variant)
    if not f32 or shared:
        assert (launches, n_exact) == (1, -1), (case, variant, launches, n_exact)
    else:
        assert launches == 2 and 0 <= n_exact <= n, (case, variant, launches, n_exact)
        if case in ALL_HANDED_OVER:
            assert n_exact == n, (case, variant, n_exact)
    aux = cache.aux(case)
    tie = _positive_shear_tie(aux, f32)
    assert tie.sum() <= NEAR_CAP * n, (case, variant, int(tie.sum()))
    call = variant + ("/ignore_nans" if ignore_nans else "")
    for min_set in (False, True):
        if min_set and ignore_nans:
            continue                                   # min_conv_properties has no mask
        got, prox = _run(cache, case, variant, ignore_nans, min_set)
        ora, prox_ora = cache.oracle(case, min_set, ignore_nans and not min_set)
        assert set(got) == set(ora), set(got) ^ set(ora)
        B = _bounds(ora, aux, f32, mu_td)
        near_ml = B.pop("melting_near")
        assert near_ml.sum() <= NEAR_CAP * n, (case, call, int(near_ml.sum()))
        B["melting_level_excuse"] = near_ml
        name = call + ("/min" if min_set else "")
        _check(case, name, got, ora, B, f"{case}/{name}: ")
        # positive_shear: equal wherever the two wind magnitudes are farther apart than their bounds
        a, b = _f64(got["positive_shear"]), np.asarray(ora["positive_shear"], np.float64)
        assert np.array_equal(np.isnan(a), np.isnan(b)), f"{case}/{name}: positive_shear NaN pattern"
        bad = np.flatnonzero(~np.isnan(b) & ~tie & (a != b))
        assert bad.size == 0, f"{case}/{name}: positive_shear differs in columns {bad[:8]}"
        if min_set:
            continue
        ex, b_ship, ship_nan_excuse = _flag_excuses(ora, B, prox_ora, tie, f32)
        for k in _lib.PROXY_FLAGS:
            g, r = _host(prox[k]).astype(bool), np.asarray(prox_ora[k]).astype(bool)
            assert ex[k].sum() <= NEAR_CAP * n, (case, name, k, int(ex[k].sum()))
            diff = np.flatnonzero((g != r) & ~ex[k])
            assert diff.size == 0, f"{case}/{name}: {k} differs from the oracle in columns {diff[:8]}"
            REPORT[f"{case} / {name} / {k}"] = (float((g != r).sum()), 0.0, int(ex[k].sum()))
        _check(case, name, prox, {"ship": prox_ora["ship"]},
               {"ship": b_ship, "ship_excuse": ex["ship"], "ship_nan_excuse": ship_nan_excuse}, f"{case}/{name}: ")
    if variant == "f32-cuda":
        # float32 NumPy and float32 CUDA tensors: the same kernels on the same values, bit for bit
        for min_set in (False, True) if not ignore_nans else (False,):
            a, pa = _run(cache, case, "f32", ignore_nans, min_set)
            b, pb = _run(cache, case, "f32-cuda", ignore_nans, min_set)
            for k in list(a) + list(pa):
                x, y = (a[k], b[k]) if k in a else (pa[k], pb[k])
                assert _same_bits(_host(x), _host(y)), (case, min_set, k)


def _same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


def test_regimes_reach_the_branches(cache):
    """The cases reach what they are here for: unbracketed 850 / 700 hPa (NaN DCI and lapse rate where the columns
    are otherwise valid), columns without a 0 C crossing, crossings below ground on the ERA5 extrapolation, several
    crossings, MU mixing ratios inside SHIP's 11-13.6 g/kg window, NaN dewpoints from q <= 0 and, masked below ground,
    columns whose mask differs between ignore_nans True and False."""
    def ora(case, ignore_nans=True):
        return cache.oracle(case, False, ignore_nans)[0]
    terrain = ora("terrain")
    assert 0.05 < np.isnan(terrain["mixed_100_dci"]).mean() < 0.9
    assert 0.02 < np.isnan(terrain["lapse_rate_700_500"]).mean() < 0.6
    assert np.isnan(ora("cold")["freezing_level"]).mean() > 0.2
    d = cache.wide("terrain_era5")
    surface = d["height_asl"][0] - d["wind_height_above_surface"][0]
    with np.errstate(invalid="ignore"):
        assert (ora("terrain_era5")["freezing_level"] < surface).sum() > 10          # below ground
    wb_cross = []
    for case in CASES:
        d = cache.wide(case)
        with np.errstate(invalid="ignore"):
            s = np.sign(d["temperature"] - 273.15)
        wb_cross.append(((s[:-1] != s[1:]) & ~np.isnan(s[:-1]) & ~np.isnan(s[1:])).sum(axis=0))
    assert (np.concatenate(wb_cross) >= 3).sum() > 10                   # inversions: several crossings
    with np.errstate(invalid="ignore"):
        mr = ora("terrain")["mu_mixing_ratio"]
        assert ((mr >= 0.011) & (mr <= 0.0136)).sum() > 20
    assert cache.oracle("terrain", False, False)[1]["proxy_SHIP_0.1"].sum() > 10
    for case in CASES:
        d = cache.wide(case)
        assert np.isnan(d["dewpoint"][-2:, 3::53]).all() and np.isnan(d["dewpoint"][-2:, 7::211]).all(), case
    masked, kept = ora("masked_era5", False), ora("masked_era5", True)
    nan_m, nan_k = np.isnan(masked["mixed_100_cape"]), np.isnan(kept["mixed_100_cape"])
    assert nan_m.mean() > 0.8 and nan_k.mean() < 0.5 and (~nan_m).sum() > 20


# ---- layouts and array types, bit for bit ------------------------------------------------------------------------------
LAYOUT_CASES = ["terrain", "terrain_era5", "masked_era5"]


def _to_layout(dat, layout, L):
    """[L, N] fields and [N] surface winds as [N, L] (vert_axis=1) or (2, L, 25, 40) (vert_axis=1); a 1-D pressure stays
    1-D."""
    out = {}
    for k, v in dat.items():
        if v.ndim == 1 and v.shape[0] == L and k == "pressure":
            out[k] = v
        elif v.ndim == 1:
            out[k] = v if layout == "NL" else v.reshape(2, 25, 40)
        elif layout == "NL":
            out[k] = np.ascontiguousarray(v.T)
        else:
            out[k] = np.ascontiguousarray(v.reshape(L, 2, 25, 40).transpose(1, 0, 2, 3))
    return out


@pytest.mark.parametrize("layout", ["NL", "4d"])
@pytest.mark.parametrize("case", LAYOUT_CASES)
def test_layouts_give_the_same_bits(cache, case, layout):
    """[L, N] (vert_axis=0) against [N, L] and (2, L, y, x) fields with vert_axis=1: every output equal bit for bit
    (the NaN mask reduces over the layout's vertical axis)."""
    assert N_COLUMNS == 2000
    dat = _inputs(cache, case, "f32")
    L = dat["temperature"].shape[0]
    lay = _to_layout(dat, layout, L)
    for min_set in (False, True):
        ref, pref = _run(cache, case, "f32", False, min_set)
        if min_set:
            got = dict(parcel.min_conv_properties(dict(lay), vert_axis=1, metpy_compat=_compat(case)))
            pgot = {}
        else:
            got = parcel.conv_properties(dict(lay), vert_axis=1, metpy_compat=_compat(case))
            pgot = dict(parcel.storm_proxies(got))
        assert set(got) == set(ref)
        for k in list(ref) + list(pref):
            a = _host(ref[k] if k in ref else pref[k])
            b = _host(got[k] if k in got else pgot[k])
            assert b.shape == ((N_COLUMNS,) if layout == "NL" else (2, 25, 40)), (k, b.shape)
            assert _same_bits(a, b.reshape(-1)), (case, layout, min_set, k)


@pytest.mark.parametrize("dtype", ["f32", "f64"])
@pytest.mark.parametrize("case", AXIS_CASES)
def test_shared_axis_column_counts(cache, case, dtype):
    """A shared 1-D pressure axis broadcasts along the vertical axis whatever the number of columns: N = 37 (as many
    columns as levels) and N = 1 equal the first 37 / 1 columns of the N = 2000 call bit for bit.  Slicing columns moves
    no bits (test_gpu_regimes.test_warp_neighbours_do_not_move_results), so a difference is a misaligned pressure."""
    dat = _inputs(cache, case, dtype)
    L = dat["temperature"].shape[0]
    assert dat["pressure"].shape == (L,) == (37,)
    for min_set in (False, True):
        ref, pref = _run(cache, case, dtype, False, min_set)
        for n in (37, 1):
            sub = {k: (v if k == "pressure" else np.ascontiguousarray(v[..., :n])) for k, v in dat.items()}
            if min_set:
                got, pgot = dict(parcel.min_conv_properties(sub, metpy_compat=_compat(case))), {}
            else:
                got = parcel.conv_properties(sub, metpy_compat=_compat(case))
                pgot = dict(parcel.storm_proxies(got))
                assert sub["dewpoint"].shape == (L, n)
            for k in list(ref) + list(pref):
                a = _host(ref[k] if k in ref else pref[k])[:n]
                b = _host(got[k] if k in got else pgot[k])
                assert _same_bits(a, b), (case, dtype, min_set, n, k)


@pytest.mark.parametrize("dtype", ["f32", "f64"])
@pytest.mark.parametrize("case", ["terrain_era5", "masked_era5"])
def test_downdraft_and_effective_on_the_shared_axis(cache, case, dtype):
    """conv_properties(downdraft=True, effective=True) on the 1-D axis: dcape and effective_inflow_* equal the
    standalone downdraft_cape and effective_inflow_layer on the dewpoint conv_properties returns, masked the same way."""
    dat = _inputs(cache, case, dtype)
    compat = _compat(case)
    d = dict(dat)
    got = parcel.conv_properties(d, metpy_compat=compat, downdraft=True, effective=True)
    td = d["dewpoint"]
    assert td.shape == dat["temperature"].shape
    ref, _ = _run(cache, case, dtype, False, False)
    for k in ref:
        assert _same_bits(_host(ref[k]), _host(got[k])), k
    p, t, q = dat["pressure"], dat["temperature"], dat["specific_humidity"]
    bad = np.isnan(td).any(0) | np.isnan(p).any() | np.isnan(t).any(0) | np.isnan(q).any(0)
    assert 0 < bad.sum() < bad.size
    dc = parcel.downdraft_cape(p, t, td, metpy_compat=compat)["dcape"]
    eff = parcel.effective_inflow_layer(p, t, td, metpy_compat=compat)
    want = {"dcape": dc, **{k: eff[k] for k in _lib.EFFECTIVE_FIELDS}}
    for k, v in want.items():
        assert _same_bits(np.where(bad, np.nan, v), _host(got[k])), k
        assert np.isfinite(_host(got[k])).sum() > 0, k
