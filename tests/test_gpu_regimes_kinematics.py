"""Storm kinematics and the effective-layer parameters on the GPU (DESIGN.md section 3.14) on the real-world column
regimes of tests/regime_columns.py, in float32 and float64, on every layout and under non-default arguments.

* The kinematics kernel on every regime of test_gpu_regimes_dcape_effective (70 and 137 model levels, 16 / 24 / 40
  per-column levels, the 37 ERA5 levels extrapolated or masked below ground, deep shared axes), with NaN surface winds,
  levels exactly at 500 / 5500 / 6000 m, profiles that end below 6 km and per-column SRH / BWD layers built from the
  effective-layer heights plus reversed, zero-depth, NaN and below-ground bounds; against kinematics_oracle on the
  same (dtype-rounded) inputs.
* The read extent of contract item 5 on the device: every level above the extent is overwritten with a height below
  the previous level's and winds of 1e4, and no output may move a bit; poisoning the extent level itself must move one.
* effective_layer_parameters in both dtypes against the oracle's composition of the library's own pieces, with the
  float32 bounds derived below and every threshold of contract item 6 treated explicitly; a from-scratch float64
  oracle on a sample of every case; a pairwise matrix of non-default arguments; layouts and xarray; and
  conv_properties(kinematics=True, effective=True) against the oracle's assembly of the same steps.
"""

import itertools

import numpy as np
import pytest
import torch

import effective_oracle as eo
import kinematics_oracle as ko
import regime_columns as rc
from oracle import parcel as op
from oracle import tables as otab
from oracle import thermo as th
from test_gpu_kinematics import _compare as kin_compare, _strided
from test_gpu_regimes_conv import CASES as CONV_CASES, _compat as conv_compat, _to_layout
from test_gpu_regimes_dcape_effective import AXIS_CASES, CASES
from xarray_parcel_b200 import _lib
import xarray_parcel_b200.parcel_functions as parcel

pytestmark = pytest.mark.gpu

ALL = CASES + AXIS_CASES
ALL_IDS = [c[0] for c in ALL]
N_COLUMNS = 2000
DTYPES = {"f32": torch.float32, "f64": torch.float64}
DEPTHS = (1000.0, 3000.0, 500.0, 6000.0)
WIND_KEYS = ("wind_height_above_surface", "wind_u", "wind_v", "surface_wind_u", "surface_wind_v")
# injected into every case: NaN surface u / v, profiles ending below 6 km, levels exactly at the Bunkers bounds
NAN_U_COLUMNS, NAN_V_COLUMNS = slice(4, None, 89), slice(45, None, 89)
SHORT_COLUMNS, SHORT_TOP = slice(6, None, 41), 5900.0
EXACT_LEVELS = {500.0: slice(11, None, 37), 5500.0: slice(23, None, 37), 6000.0: slice(30, None, 37)}

# ---- bounds ----------------------------------------------------------------------------------------------------------
# U: float32 unit roundoff (one rounding of x moves it by at most U |x|).  F64_NOISE: float64 evaluations of the same
# values in another operation order.  SECOND_ORDER covers the O(U^2) terms of the first-order propagations.
U = 2.0 ** -24
F64_NOISE = 1e-12
SECOND_ORDER = 1.01
# columns allowed on the other side of a discontinuous threshold (EBWD 10 / 12.5 m/s) than the oracle
JUMP_CAP = 0.005
# the from-scratch oracle, relative to 1 + |x|: EBWD and the composites read the library's ML / MU lifts.  On a shared
# 37-level axis those carry the float32 sweep's rounding (profile rows within 3e-6, test_gpu_regimes_conv PROFILE_RTOL):
# an EL pressure off by 3e-6 moves its height by up to |dz / d ln p| * 3e-6 < 1e4 m * 3e-6 = 0.03 m, and EBWD by the wind
# shear over that, which 1e-6 does not cover; the bound of test_gpu_kinematics' composition test
SCRATCH_RTOL = 1e-4
SCRATCH_N = 200


def _np(x):
    return np.asarray(x.cpu().numpy() if isinstance(x, torch.Tensor) else x, dtype=np.float64)


def _bits(x):
    x = np.ascontiguousarray(x.cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x))
    return x.dtype, x.shape, x.tobytes()


def _mover(case):
    return "right" if ALL_IDS.index(case) % 2 == 0 else "left"


# ---- fixtures and inputs -----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    c = _lib.get_context(0)
    if not c.tables_loaded():
        c.tables_build()
    return c


@pytest.fixture(scope="module")
def gpu_tables(ctx):
    idx, cur = ctx.tables_get()
    pl, tl = otab.default_grids()
    return otab.AdiabatTables(pl, tl, idx, cur)


def _inject(f):
    """The kinematics edges every case carries (in place, float32): NaN surface winds, profiles ending at SHORT_TOP
    (winds NaN above) and a kept level moved onto 500 / 5500 / 6000 m exactly (it stays between its neighbours)."""
    h, u, v = f["wind_height_above_surface"], f["wind_u"], f["wind_v"]
    f["surface_wind_u"][NAN_U_COLUMNS] = np.nan
    f["surface_wind_v"][NAN_V_COLUMNS] = np.nan
    with np.errstate(invalid="ignore"):
        short = np.zeros(h.shape, dtype=bool)
        short[:, SHORT_COLUMNS] = h[:, SHORT_COLUMNS] >= SHORT_TOP
    u[short] = np.nan
    v[short] = np.nan
    for target, cols in EXACT_LEVELS.items():
        for c in range(h.shape[1])[cols]:
            with np.errstate(invalid="ignore"):
                ks = np.flatnonzero(np.isfinite(u[:, c]) & np.isfinite(v[:, c]) & (h[:, c] >= target))
            if ks.size:
                h[ks[0], c] = target
    return f


def _layers(extra, n, seed):
    """(SRH layer, BWD layer) [N] float32: the effective layer [z_base, z_top] and EBWD's [max(z_base, 0), half the MU
    EL height above it] where the column has them (random layers elsewhere), then reversed, zero-depth, NaN-bottom,
    NaN-top, below-ground and entirely below-ground bounds in every 23rd column."""
    rng = np.random.default_rng(seed)
    fb = rng.uniform(-400.0, 3000.0, n)
    ft = fb + rng.uniform(-200.0, 5000.0, n)
    zb, zt, zel = extra["z_base"], extra["z_top"], extra["z_el"]
    has = np.isfinite(zb)
    sb, st = np.where(has, zb, fb), np.where(has, zt, ft)
    zb0 = np.maximum(sb, 0.0)
    bb, bt = zb0, np.where(has & np.isfinite(zel), zb0 + (zel - zb0) / 2.0, ft)
    out = []
    for j, (b, t) in enumerate(((sb, st), (bb, bt))):
        b, t = b.copy(), t.copy()
        o = 7 * j
        b[o::23], t[o::23] = t[o::23].copy(), b[o::23].copy()          # reversed
        t[o + 1::23] = b[o + 1::23]                                    # zero depth
        b[o + 2::23] = np.nan
        t[o + 3::23] = np.nan
        b[o + 4::23] = -250.0                                          # bottom below ground
        b[o + 5::23], t[o + 5::23] = -300.0, -100.0                    # the whole layer below ground: [0, 0]
        out.append((b.astype(np.float32), t.astype(np.float32)))
    return out


class _Cache:
    """Inputs, library pieces and oracle results per case, computed once for the module."""

    def __init__(self, tables):
        self.tables, self.store = tables, {}

    def get(self, key, make):
        if key not in self.store:
            self.store[key] = make()
        return self.store[key]

    def inputs(self, case):
        """float32 (p, T, Td) and the wind fields (WIND_KEYS) of a case."""
        def make():
            i = ALL_IDS.index(case)
            _, regime, kw = ALL[i]
            p, t, td, p0 = rc.columns(regime, N_COLUMNS, seed=900 + i, **kw)
            f = _inject(rc.conv_fields(p, t, td, p0, seed=950 + i))
            return dict(f, dewpoint=td)
        return self.get(("inputs", case), make)

    def wide(self, case):
        return self.get(("wide", case), lambda: {k: v.astype(np.float64) for k, v in self.inputs(case).items()})

    def opts(self, metpy_compat="1.4.1"):
        return op.Options(op.MoistLapseLUT(self.tables), metpy_compat=metpy_compat)

    def effective(self, ctx, case, dt):
        """(library result, oracle outputs, scales, pieces + heights) of effective_layer_parameters on the case."""
        def make():
            d, w = self.inputs(case), self.wide(case)
            ty = np.float32 if dt == "f32" else np.float64
            args = [d[k].astype(ty) for k in ("pressure", "temperature", "dewpoint") + WIND_KEYS]
            r = parcel.effective_layer_parameters(*args, mover=_mover(case))
            pieces = _pieces(ctx, *args[:3], {})
            want, scale, extra = ko.effective_layer_parameters(
                w["pressure"], w["temperature"], w["dewpoint"], *[w[k] for k in WIND_KEYS], self.opts(),
                _lib.MOVERS[_mover(case)], pieces=pieces)
            return r, want, scale, extra
        return self.get(("effective", case, dt), make)

    def layers(self, ctx, case):
        return self.get(("layers", case), lambda: _layers(self.effective(ctx, case, "f64")[3], N_COLUMNS,
                                                           ALL_IDS.index(case)))

    def kinematics(self, ctx, case):
        """The oracle's storm_kinematics of the full call (motion, DEPTHS, both layers) on the float32 inputs."""
        def make():
            w = self.wide(case)
            sl, bl = self.layers(ctx, case)
            lay = lambda x: tuple(a.astype(np.float64) for a in x)            # noqa: E731
            return ko.storm_kinematics(*[w[k] for k in WIND_KEYS], _lib.MOVERS[_mover(case)], DEPTHS, lay(sl),
                                       lay(bl))
        return self.get(("kinematics", case), make)


@pytest.fixture(scope="module")
def cache(gpu_tables):
    return _Cache(gpu_tables)


OPTION_KEYS = ("virtual_temperature_correction", "lcl_interp", "metpy_compat")


def _pieces(ctx, p, t, td, args):
    """The pieces effective_layer_parameters composes (its base / top and the ML / MU lift values), from the library's
    own calls with ``args`` (the composition's keywords), as float64 NumPy."""
    dt = torch.float32 if np.asarray(t).dtype == np.float32 else torch.float64
    dev = [torch.from_numpy(np.ascontiguousarray(x)).to(dt).cuda() for x in (p, t, td)]
    opt = {k: args[k] for k in OPTION_KEYS if k in args}
    mud, mld = args.get("most_unstable_depth", 300.0), args.get("mixed_layer_depth", 100.0)
    eff = ctx.effective_inflow_layer(*dev, options=_lib.make_options(most_unstable_depth=mud, **opt),
                                     min_cape=args.get("min_cape", 100.0), min_cin=args.get("min_cin", -250.0))
    lifted = ctx.cape_cin(*dev, kinds=("ml", "mu"), options=_lib.make_options(
        mixed_layer_depth=mld, most_unstable_depth=mud, **opt))
    ml, mu = lifted["ml"], lifted["mu"]
    return {"effective_inflow_base": _np(eff["effective_inflow_base"]),
            "effective_inflow_top": _np(eff["effective_inflow_top"]), "mu_cape": _np(mu["cape"]),
            "mu_el_pressure": _np(mu["el_pressure"]), "ml_cape": _np(ml["cape"]), "ml_cin": _np(ml["cin"]),
            "ml_lcl_pressure": _np(ml["lcl_pressure"])}


# ---- the effective-layer bounds ----------------------------------------------------------------------------------------
def _wind_slope(H, U_, V, SU, SV, zc, dz):
    """Per column: the steepest |du| + |dv| per metre of the profile segments that meet [zc - dz, zc + dz], and the
    profile's highest point (NaN: no profile)."""
    n = H.shape[1]
    slope, ztop = np.zeros(n), np.full(n, np.nan)
    for c in range(n):
        prof = ko.profile(H[:, c], U_[:, c], V[:, c], SU[c], SV[c], np.nan)
        if prof is None:
            continue
        z, u, v = prof
        ztop[c] = z[-1]
        if not np.isfinite(zc[c]) or z.size < 2:
            continue
        s = (np.abs(np.diff(u)) + np.abs(np.diff(v))) / np.diff(z)
        meet = (z[1:] >= zc[c] - dz[c]) & (z[:-1] <= zc[c] + dz[c])
        slope[c] = s[meet].max(initial=0.0)
    return slope, ztop


def _eff_bounds(want, scale, extra, w, f32, mover):
    """Per-column bounds of |library - oracle| for ESRH, EBWD, SCP and STP when the library's pieces are the oracle's
    pieces, and the columns excused at the two discontinuous thresholds.  ``eps``: U for float32 results, F64_NOISE for
    float64.

    * ESRH: the layer [z_base, z_top] is the base and top level's own heights in both (xp_interp_levels returns a
      level's own height at its pressure, pinned below), so the kinematics bound: 1e-9 of the term scale plus the
      output rounding.
    * EBWD = |V(t) - V(zb0)| with t = zb0 + (z_el - zb0) / 2 evaluated in the input dtype: z_el is one rounding of the
      float64 interpolation (eps |z_el|), the difference and the sum round once each, halving is exact, so
      |dt| <= eps (|z_el| / 2 + |z_el - zb0| / 2 + |t|).  V is linear in height on each segment: |dV| <= slope * |dt|
      over the segments within dt of t; plus the kinematics bound.  Where t lies within dt of the profile's top, the
      layer may reach or miss the top, and where t lies within dt of zb0 it may be reversed or not: such columns are
      excused (counted with the jumps).
    * SCP = (mucape / 1000) (esrh / 50) t_b: mucape is the piece itself (exact); t_b is ebwd / 20 between 10 and 20
      m/s, clipped to 1 above 20 (continuous, 1-Lipschitz in ebwd / 20), so |dt_b| <= B_ebwd / 20 there with no excuse;
      0 below 10 m/s (a jump of 0.5).  STP likewise with t_b jumping at 12.5 m/s and clipped at 30 (continuous), t_lcl
      continuous in the LCL height (one rounding of its interpolation: |dt_lcl| <= eps |z_lcl| / 1000, no excuse at
      1000 / 2000 m) and t_cin exact (mlcin is the piece).  max(0, x) is 1-Lipschitz.  Products propagate to first
      order with SECOND_ORDER, plus one output rounding.
    * At a jump: a column may differ only if its EBWD lies within B_ebwd of 10 (SCP) or 12.5 (STP) m/s."""
    eps = U if f32 else F64_NOISE
    with np.errstate(invalid="ignore"):
        esrh, ebwd = want["effective_srh"], want["effective_bulk_wind_difference"]
        b_esrh = 1e-9 * scale["effective_srh"] + eps * np.abs(esrh)
        zb0, zel, zlcl = np.maximum(extra["z_base"], 0.0), extra["z_el"], extra["z_lcl"]
        t = zb0 + (zel - zb0) / 2.0
        dt = SECOND_ORDER * eps * (np.abs(zel) / 2 + np.abs(zel - zb0) / 2 + np.abs(t))
        slope, ztop = _wind_slope(w["wind_height_above_surface"], w["wind_u"], w["wind_v"], w["surface_wind_u"],
                                  w["surface_wind_v"], t, dt)
        b_ebwd = SECOND_ORDER * slope * dt + 1e-9 * scale["effective_bulk_wind_difference"] + eps * np.abs(ebwd)
        # t within dt of the profile's top (the layer may reach it or not) or of zb0 (it may turn reversed)
        top_edge = np.isfinite(extra["z_base"]) & ((np.abs(t - ztop) <= dt) | ((np.abs(t - zb0) <= dt) & (t != zb0)))
        no_layer = np.isnan(extra["effective_inflow_base"])
        s = np.where(no_layer, 0.0, esrh) * mover
        bs = np.where(no_layer, 0.0, b_esrh)
        bb = np.where(no_layer, 0.0, b_ebwd)
        b = np.where(no_layer, 0.0, ebwd)
        # SCP
        tb = np.where(b < 10.0, 0.0, np.where(b > 20.0, 1.0, b / 20.0))
        dtb = np.where(b > 20.0 + bb, 0.0, bb / 20.0)
        mu = np.abs(extra["mu_cape"]) / 1000.0
        scp = want["supercell_composite_parameter"]
        b_scp = SECOND_ORDER * mu * (bs / 50.0 * np.abs(tb) + (np.abs(s) + bs) / 50.0 * dtb) + eps * np.abs(scp)
        jump_scp = np.abs(b - 10.0) <= bb
        # STP
        tb = np.where(b < 12.5, 0.0, np.where(b > 30.0, 1.5, b / 20.0))
        dtb = np.where(b > 30.0 + bb, 0.0, bb / 20.0)
        lcl = zlcl
        tl = np.where(lcl < 1000.0, 1.0, np.where(lcl > 2000.0, 0.0, (2000.0 - lcl) / 1000.0))
        dtl = eps * np.abs(lcl) / 1000.0
        cin = extra["ml_cin"]
        tc = np.abs(np.where(cin > -50.0, 1.0, np.where(cin < -200.0, 0.0, (cin + 200.0) / 150.0)))
        ml = np.abs(extra["ml_cape"]) / 1500.0
        stp = want["significant_tornado_parameter"]
        b_stp = SECOND_ORDER * ml * tc * (bs / 150.0 * np.abs(tb) * tl + (np.abs(s) + bs) / 150.0 *
                                           (dtb * (tl + dtl) + np.abs(tb) * dtl)) + eps * np.abs(stp)
        jump_stp = np.abs(b - 12.5) <= bb
    return ({"effective_srh": b_esrh, "effective_bulk_wind_difference": b_ebwd, "supercell_composite_parameter": b_scp,
             "significant_tornado_parameter": b_stp},
            {"effective_bulk_wind_difference": top_edge, "effective_srh": np.zeros_like(top_edge),
             "supercell_composite_parameter": jump_scp | top_edge,
             "significant_tornado_parameter": jump_stp | top_edge})


def _check_eff(got, want, bounds, excuse, what, mask=None):
    """NaN patterns identical (except excused columns) and |got - want| <= bound for the four effective-layer
    parameters; ``mask``: columns set to NaN on both sides first.  Returns {output: (excused, max err / bound)}."""
    stat = {}
    for k in _lib.EFFECTIVE_PARAMETER_FIELDS:
        g, w_ = _np(got[k]), np.array(want[k], np.float64)
        if mask is not None:
            w_[mask] = np.nan
        ex = excuse[k] if mask is None else excuse[k] & ~mask
        mis = np.flatnonzero((np.isnan(g) != np.isnan(w_)) & ~ex)
        assert mis.size == 0, f"{what}{k}: NaN pattern differs in columns {mis[:8]} (got {g[mis[:4]]}, want {w_[mis[:4]]})"
        ok = ~np.isnan(g) & ~np.isnan(w_) & ~ex
        err = np.where(ok, np.abs(np.where(ok, g, 0.0) - np.where(ok, w_, 0.0)), 0.0)
        with np.errstate(invalid="ignore", divide="ignore"):
            over = np.flatnonzero(ok & ~(err <= bounds[k]))
            ratio = float(np.max(np.where(ok & (bounds[k] > 0), err / bounds[k], 0.0), initial=0.0))
        assert over.size == 0, (f"{what}{k}: {over.size} columns outside the bound, e.g. "
                                f"{[(int(i), float(g[i]), float(w_[i]), float(bounds[k][i])) for i in over[:4]]}")
        stat[k] = (int(ex.sum()), ratio)
    return stat


# ---- 1. the kinematics kernel on every regime ---------------------------------------------------------------------------
def _dev(arrays, dtype):
    return [torch.from_numpy(np.ascontiguousarray(x)).to(dtype).cuda() for x in arrays]


def _profile_top(w):
    """Per column: the highest kept profile height (0 with none)."""
    h, u, v = w["wind_height_above_surface"], w["wind_u"], w["wind_v"]
    with np.errstate(invalid="ignore"):
        kept = np.isfinite(h) & np.isfinite(u) & np.isfinite(v) & (h > 0)
    return np.where(kept, h, 0.0).max(axis=0)


@pytest.mark.parametrize("dt", list(DTYPES))
@pytest.mark.parametrize("case", ALL_IDS)
def test_kinematics_regimes_against_oracle(ctx, cache, case, dt):
    """The full call (motion, four depths, per-column SRH and BWD layers) against the oracle on the float32 inputs
    both dtypes read; NaN patterns identical."""
    dtype = DTYPES[dt]
    d = cache.inputs(case)
    sl, bl = cache.layers(ctx, case)
    z, u, v, su, sv = _dev([d[k] for k in WIND_KEYS], dtype)
    got = ctx.storm_kinematics(z, u, v, su, sv, mover=_mover(case), depths=DEPTHS, srh_layer=tuple(_dev(sl, dtype)),
                               bwd_layer=tuple(_dev(bl, dtype)))
    want, scale = cache.kinematics(ctx, case)
    kin_compare(got, want, scale, dt == "f32")
    w = cache.wide(case)
    srh = _np(got["srh_0_3000m"])
    print(f"REGIME_STAT kinematics {case} {dt} mover={_mover(case)} nan_fraction={np.isnan(srh).mean():.4f} "
          f"below_6km_fraction={(_profile_top(w) < 6000.0).mean():.4f} "
          f"srh_layer_nan_fraction={np.isnan(_np(got['srh_layer'])).mean():.4f}")
    assert np.isfinite(srh).mean() > 0.8


def test_cases_reach_the_kinematics_branches(ctx, cache):
    """The cases reach what they are here for: levels dropped below ground, masked (NaN wind) levels, profiles ending
    below 6 km, NaN surface winds, kept levels exactly at 500 / 5500 / 6000 m, effective bases below ground (EBWD's
    clamp to 0), and effective layers with a weak shear (0 < EBWD < 10 m/s, SCP's zero branch)."""
    below = masked = short = nan_sfc = 0
    exact = {t: 0 for t in EXACT_LEVELS}
    for case in ALL_IDS:
        w = cache.wide(case)
        h, u = w["wind_height_above_surface"], w["wind_u"]
        with np.errstate(invalid="ignore"):
            below += int((np.isfinite(h) & np.isfinite(u) & (h <= 0)).sum())
            masked += int((np.isfinite(h) & np.isnan(u)).sum())
            for t in exact:
                exact[t] += int(((h == t) & np.isfinite(u)).sum())
        short += int(((_profile_top(w) < 6000.0) & np.isfinite(w["surface_wind_u"] + w["surface_wind_v"])).sum())
        nan_sfc += int(np.isnan(w["surface_wind_u"] + w["surface_wind_v"]).sum())
    assert below > 1000 and masked > 1000 and short > 500 and nan_sfc > 500, (below, masked, short, nan_sfc)
    assert min(exact.values()) > 500, exact
    zb_neg = weak = 0
    for case in ALL_IDS:
        _, want, _, extra = cache.effective(ctx, case, "f64")
        with np.errstate(invalid="ignore"):
            zb_neg += int((extra["z_base"] < 0).sum())
            ebwd = want["effective_bulk_wind_difference"]
            weak += int(((ebwd > 0) & (ebwd < 10.0) & (np.abs(want["effective_srh"]) > 1.0) &
                         (extra["mu_cape"] > 100.0)).sum())
    print(f"REGIME_STAT branches below_ground_levels={below} masked_levels={masked} short_columns={short} "
          f"nan_surface_wind={nan_sfc} exact={exact} base_below_ground={zb_neg} weak_shear={weak}")
    assert zb_neg > 20 and weak > 20, (zb_neg, weak)


# ---- 2. the device read extent -----------------------------------------------------------------------------------------
def _top_needed(sl, bl, motion, srh_layer, bwd_layer):
    """Per column: the highest bound the call needs (item 5), -inf when it needs none."""
    tops = [np.full(sl[0].shape, 6000.0 if motion else -np.inf)]
    for use, (b, t) in ((srh_layer, sl), (bwd_layer, bl)):
        if use:
            b, t = np.maximum(b.astype(np.float64), 0.0), np.maximum(t.astype(np.float64), 0.0)
            with np.errstate(invalid="ignore"):
                tops.append(np.where(np.isfinite(b) & np.isfinite(t) & (t >= b), t, -np.inf))
    return np.max(tops, axis=0)


def _extent(w, top):
    """Per column: the last level item 5 reads -- the first kept level at or above ``top``, or the first kept level
    whose height does not increase (the column stops there) -- and -1 when nothing is read (a NaN surface wind, or no
    bound above the surface).  L - 1 when the column never reaches ``top``: it reads every level.  Also returns the
    highest kept height before each level and up to each level (0 with none)."""
    h, u, v = w["wind_height_above_surface"], w["wind_u"], w["wind_v"]
    L, n = h.shape
    with np.errstate(invalid="ignore"):
        kept = np.isfinite(h) & np.isfinite(u) & np.isfinite(v) & (h > 0)
    run = np.maximum.accumulate(np.where(kept, h, 0.0), axis=0)
    prev = np.vstack([np.zeros((1, n)), run[:-1]])
    with np.errstate(invalid="ignore"):
        stop = kept & ((h >= top[None, :]) | (h <= prev))
    ext = np.where(stop.any(axis=0), np.argmax(stop, axis=0), L - 1)
    none = np.isnan(w["surface_wind_u"]) | np.isnan(w["surface_wind_v"]) | ~(top > 0)
    return np.where(none, -1, ext), prev, run


EXTENT_VARIANTS = ["all", "srh_only", "bwd_only", "strided"]


@pytest.mark.parametrize("variant", EXTENT_VARIANTS)
@pytest.mark.parametrize("case", ALL_IDS)
def test_device_read_extent(ctx, cache, case, variant):
    """Levels above each column's extent are overwritten, inside the arrays, with a height below the previous kept
    level's (a read would end the column as non-increasing: NaN) and winds of 1e4: every output must stay bit-identical.
    Poisoning the extent level itself must change some output.  ``all``: motion, depths and both layers; ``srh_only``:
    the SRH outputs only (the motion outputs NULL, still computed for them; the BWD layer unread); ``bwd_only``: the
    BWD layer alone (no motion, a per-column extent); ``strided``: ``all`` through a level pitch wider than N."""
    i = ALL_IDS.index(case)
    dtype = torch.float32 if i % 2 == 0 else torch.float64
    d, w = cache.inputs(case), cache.wide(case)
    sl, bl = cache.layers(ctx, case)
    srh_names = [f"srh_0_{x:g}m" for x in DEPTHS]
    kw = dict(mover=_mover(case), depths=DEPTHS, srh_layer=tuple(_dev(sl, dtype)), bwd_layer=tuple(_dev(bl, dtype)))
    motion, use_s, use_b = True, True, True
    if variant == "srh_only":
        kw["outputs"] = srh_names + ["srh_layer"]
        use_b = False
    elif variant == "bwd_only":
        kw = dict(bwd_layer=kw["bwd_layer"], outputs=list(_lib.BWD_FIELDS))
        motion = use_s = False
    top = _top_needed(sl, bl, motion, use_s, use_b)
    ext, prev, run_max = _extent(w, top)
    L, n = w["wind_height_above_surface"].shape
    cols = np.arange(n)

    def run(h, u, v):
        z, uu, vv, su, sv = _dev([h, u, v, d["surface_wind_u"], d["surface_wind_v"]], dtype)
        if variant == "strided":
            z, uu, vv = _strided(z), _strided(uu), _strided(vv)
            assert uu.stride(0) == n + 37
        return ctx.storm_kinematics(z, uu, vv, su, sv, **kw)

    h0, u0, v0 = [d[k].copy() for k in WIND_KEYS[:3]]
    ref = run(h0, u0, v0)
    above = np.arange(L)[:, None] > ext[None, :]
    poison_h = (np.where(ext >= 0, run_max[np.clip(ext, 0, None), cols], 0.0) / 2.0).astype(np.float32)
    h1, u1, v1 = h0.copy(), u0.copy(), v0.copy()
    h1[above] = np.broadcast_to(poison_h, (L, n))[above]
    u1[above] = 1e4
    v1[above] = 1e4
    got = run(h1, u1, v1)
    for k in ref:
        assert _bits(got[k]) == _bits(ref[k]), (case, variant, k)
    poisoned = int(above.sum())
    assert poisoned > (0.05 if variant == "bwd_only" else 0.1) * L * n, poisoned
    # the extent level itself: the same poison must move some output
    at = (ext >= 0) & (ext < L)
    k_at = np.clip(ext, 0, None)
    h2, u2, v2 = h0.copy(), u0.copy(), v0.copy()
    h2[k_at[at], cols[at]] = (prev[k_at[at], cols[at]] / 2.0).astype(np.float32)
    u2[k_at[at], cols[at]] = 1e4
    v2[k_at[at], cols[at]] = 1e4
    bite = run(h2, u2, v2)
    moved = 0
    for k in ref:
        a, b = _np(bite[k]), _np(ref[k])
        moved += int(((a != b) & ~(np.isnan(a) & np.isnan(b))).sum())
    assert moved > 0.1 * n, (case, variant, moved)
    print(f"REGIME_STAT extent {case} {variant} levels_poisoned={poisoned / (L * n):.3f} "
          f"reads_all_levels={(ext == L - 1).mean():.4f} outputs_moved_at_extent={moved}")


# ---- 3. effective_layer_parameters in both dtypes on every case ----------------------------------------------------------
@pytest.mark.parametrize("dt", list(DTYPES))
@pytest.mark.parametrize("case", ALL_IDS)
def test_effective_layer_parameters_regimes(ctx, cache, case, dt):
    """Against the oracle's composition of the library's own pieces, in the input dtype: base / top equal
    effective_inflow_layer's bits, the height at the base equals the base level's own height bit for bit, float32 NumPy
    equals float32 CUDA tensors, and ESRH, EBWD, SCP and STP lie within _eff_bounds (jump columns counted, capped)."""
    dtype = DTYPES[dt]
    f32 = dt == "f32"
    ty = np.float32 if f32 else np.float64
    d, w = cache.inputs(case), cache.wide(case)
    r, want, scale, extra = cache.effective(ctx, case, dt)
    P, T, D = [d[k].astype(ty) for k in ("pressure", "temperature", "dewpoint")]
    eff = parcel.effective_inflow_layer(P, T, D)
    for k in _lib.EFFECTIVE_FIELDS:
        assert _bits(r[k]) == _bits(eff[k]), k
        assert np.asarray(r[k]).dtype == ty
    # the height at the base is the base level's own height (xp_interp_levels' contract)
    p_d, h_d = _dev([P, d["wind_height_above_surface"]], dtype)
    base = np.asarray(r["effective_inflow_base"])
    (zb,) = ctx.interp_levels(p_d, [h_d], torch.from_numpy(base).cuda(), log=True)
    zb = zb.cpu().numpy()
    p2 = np.broadcast_to(P.reshape(P.shape[0], -1), T.shape)
    has = np.isfinite(base)
    k_base = np.argmax(p2 == base[None, :], axis=0)
    assert (p2[k_base[has], np.flatnonzero(has)] == base[has]).all()
    h_at = d["wind_height_above_surface"].astype(ty)[k_base, np.arange(T.shape[1])]
    assert _bits(zb[has]) == _bits(h_at[has]) and np.isnan(zb[~has]).all()
    if f32:
        cuda = parcel.effective_layer_parameters(*_dev([d[k] for k in ("pressure", "temperature", "dewpoint") +
                                                         WIND_KEYS], torch.float32), mover=_mover(case))
        for k in r:
            assert _bits(r[k]) == _bits(cuda[k]), k
    bounds, excuse = _eff_bounds(want, scale, extra, w, f32, _lib.MOVERS[_mover(case)])
    n = T.shape[1]
    for k in ("supercell_composite_parameter", "significant_tornado_parameter"):
        assert excuse[k].sum() <= JUMP_CAP * n, (k, int(excuse[k].sum()))
    stat = _check_eff(r, want, bounds, excuse, f"{case}/{dt}: ")
    print(f"REGIME_STAT effective_params {case} {dt} mover={_mover(case)} layer_fraction={has.mean():.3f} "
          + " ".join(f"{k}:excused={e},err/bound={q:.2g}" for k, (e, q) in stat.items()))


# ---- 4. the from-scratch oracle on a sample of every case ---------------------------------------------------------------
def _near_threshold(extra, P, T, D, min_cape=100.0, min_cin=-250.0):
    """Columns with a level parcel whose CAPE / CIN lies within 1e-6 (relative, at least 1e-6 J/kg) of the
    thresholds (CAPE only when min_cape > 0), or a saturated valid level (T == Td, the LCL is the level itself): the effective layer may differ."""
    cape, cin = extra["level_parcel_cape"], extra["level_parcel_cin"]
    with np.errstate(invalid="ignore"):
        tol = np.maximum(np.abs(cape), 1.0) * 1e-6
        near = np.abs(cin - min_cin) < np.maximum(np.abs(cin), 1.0) * 1e-6
        if min_cape > 0:                               # CAPE >= 0: with min_cape <= 0 its test cannot flip
            near |= np.abs(cape - min_cape) < tol
    return (near | (eo.valid_levels(P, T, D) & (T == D))).any(axis=0)


def _scratch_compare(got, want, scale, extra, P, T, D, what, min_cape=100.0, min_cin=-250.0):
    """Base and top exactly the oracle's except on near-threshold columns (counted, < 5 %); on the others ESRH to the
    kinematics bound (same layer), EBWD, SCP and STP to SCRATCH_RTOL (1 + |x|), with columns whose EBWD lies within
    that of a jump excused (counted)."""
    near = _near_threshold(extra, P, T, D, min_cape, min_cin)
    same = np.ones(near.shape, dtype=bool)
    for k in _lib.EFFECTIVE_FIELDS:
        g = _np(got[k])
        same &= (g == want[k]) | (np.isnan(g) & np.isnan(want[k]))
    assert (same | near).all(), (what, np.flatnonzero(~(same | near))[:8])
    assert near.mean() < 0.05, (what, near.mean())
    ebwd = want["effective_bulk_wind_difference"]
    with np.errstate(invalid="ignore"):
        jump = (np.abs(ebwd - 10.0) <= SCRATCH_RTOL * 11.0) | (np.abs(ebwd - 12.5) <= SCRATCH_RTOL * 13.5)
    worst = {}
    for k in _lib.EFFECTIVE_PARAMETER_FIELDS:
        g, w_ = _np(got[k])[same], want[k][same]
        assert np.array_equal(np.isnan(g), np.isnan(w_)), (what, k)
        if k == "effective_srh":
            tol = 1e-9 * scale[k][same]
        else:
            tol = SCRATCH_RTOL * (1.0 + np.abs(w_))
        ok = ~np.isnan(w_)
        if k in _lib.COMPOSITE_FIELDS:
            ok &= ~jump[same]
        err = np.abs(np.where(ok, g - w_, 0.0))
        bad = np.flatnonzero(ok & ~(err <= tol))
        assert bad.size == 0, (what, k, [(int(i), float(g[i]), float(w_[i])) for i in bad[:5]])
        worst[k] = float(np.max(np.where(ok, err / (1.0 + np.abs(w_)), 0.0), initial=0.0))
    return int(near.sum()), int(jump.sum()), worst


@pytest.mark.parametrize("case", ALL_IDS)
def test_effective_from_scratch_oracle(ctx, cache, case):
    """float64, SCRATCH_N columns per case: the oracle computes the whole composition (its own effective layer and
    lifts); near-threshold columns are excused and counted."""
    d = cache.wide(case)
    cols = np.linspace(0, N_COLUMNS - 1, SCRATCH_N).astype(int)
    P = d["pressure"] if d["pressure"].ndim == 1 else np.ascontiguousarray(d["pressure"][:, cols])
    sub = {k: np.ascontiguousarray(d[k][..., cols]) for k in ("temperature", "dewpoint") + WIND_KEYS}
    T, D = sub["temperature"], sub["dewpoint"]
    winds = [sub[k] for k in WIND_KEYS]
    r = parcel.effective_layer_parameters(P, T, D, *winds, mover=_mover(case))
    want, scale, extra = cache.get(("scratch", case), lambda: ko.effective_layer_parameters(
        P, T, D, *winds, cache.opts(), _lib.MOVERS[_mover(case)]))
    near, jump, worst = _scratch_compare(r, want, scale, extra, P, T, D, case)
    print(f"REGIME_STAT scratch {case} near_threshold={near} jump_excused={jump} "
          + " ".join(f"{k}:max_rel={v:.1e}" for k, v in worst.items()))


# ---- 5. non-default arguments --------------------------------------------------------------------------------------------
ARG_NAMES = ("min_cape", "min_cin", "most_unstable_depth", "mixed_layer_depth", "virtual_temperature_correction",
             "lcl_interp", "metpy_compat", "mover")
DEFAULTS = (100, -250, 300, 100, True, "log", "1.4.1", "right")
NON_DEFAULT = {"min_cape": (0, 250), "min_cin": (-50,), "most_unstable_depth": (200, 400),
               "mixed_layer_depth": (50, 150), "virtual_temperature_correction": (False,), "lcl_interp": ("linear",),
               "metpy_compat": ("1.6.2",), "mover": ("left",)}
# every pair of values of every two arguments (the defaults included) meets in some row; the first row is the default
PAIRWISE = [
    (100, -250, 300, 100, True, "log", "1.4.1", "right"),
    (100, -50, 200, 50, False, "linear", "1.6.2", "left"),
    (0, -250, 400, 150, True, "log", "1.6.2", "left"),
    (250, -50, 400, 150, False, "linear", "1.4.1", "right"),
    (0, -250, 200, 50, True, "linear", "1.4.1", "right"),
    (250, -50, 300, 100, False, "log", "1.6.2", "left"),
    (0, -250, 300, 100, False, "linear", "1.4.1", "left"),
    (250, -250, 200, 50, True, "log", "1.6.2", "right"),
    (100, -50, 300, 150, True, "log", "1.4.1", "right"),
    (100, -250, 400, 100, True, "log", "1.4.1", "right"),
    (0, -50, 300, 50, True, "log", "1.4.1", "right"),
    (100, -250, 200, 100, True, "log", "1.4.1", "right"),
    (100, -250, 200, 150, True, "log", "1.4.1", "right"),
    (100, -250, 400, 50, True, "log", "1.4.1", "right"),
]
ARG_CASES = ("terrain_era5", "moist_heat")          # one shared ERA5 axis, one per-column model-level case
ARG_N = 150


def test_pairwise_table_covers_every_pair():
    values = {a: (dv,) + NON_DEFAULT[a] for a, dv in zip(ARG_NAMES, DEFAULTS)}
    assert PAIRWISE[0] == DEFAULTS
    for (i, a), (j, b) in itertools.combinations(enumerate(ARG_NAMES), 2):
        seen = {(row[i], row[j]) for row in PAIRWISE}
        assert seen == set(itertools.product(values[a], values[b])), (a, b)


def _arg_inputs(cache, case, ty, n=ARG_N):
    d = cache.inputs(case)
    cols = np.linspace(0, N_COLUMNS - 1, n).astype(int)
    p = d["pressure"] if d["pressure"].ndim == 1 else d["pressure"][:, cols]
    sub = [np.ascontiguousarray(x).astype(ty) for x in
           [p] + [d[k][..., cols] for k in ("temperature", "dewpoint") + WIND_KEYS]]
    return sub


def _split(row):
    a = dict(zip(ARG_NAMES, row))
    mover = a.pop("mover")
    return a, mover


@pytest.mark.parametrize("row", range(len(PAIRWISE)))
@pytest.mark.parametrize("case", ARG_CASES)
def test_arguments_pairwise_against_oracle(ctx, cache, case, row):
    """Each row's arguments in float64 against the from-scratch oracle given the same arguments, and in float32
    against the oracle's composition of the library's pieces made with them."""
    args, mover = _split(PAIRWISE[row])
    kin = {k: args[k] for k in ("virtual_temperature_correction", "lcl_interp")}
    core = {k: args[k] for k in ("min_cape", "min_cin", "most_unstable_depth", "mixed_layer_depth")}
    x64 = _arg_inputs(cache, case, np.float64)
    r = parcel.effective_layer_parameters(*x64, mover=mover, **args)
    opts = cache.opts(args["metpy_compat"])
    want, scale, extra = cache.get(("arg_scratch", case, row), lambda: ko.effective_layer_parameters(
        *x64, opts, _lib.MOVERS[mover], **core, **kin))
    near, jump, worst = _scratch_compare(r, want, scale, extra, *x64[:3], f"{case}/row {row}",
                                         args["min_cape"], args["min_cin"])
    x32 = _arg_inputs(cache, case, np.float32)
    r32 = parcel.effective_layer_parameters(*x32, mover=mover, **args)
    pieces = _pieces(ctx, *x32[:3], args)
    w32 = [x.astype(np.float64) for x in x32]
    want32, scale32, extra32 = ko.effective_layer_parameters(*w32, opts, _lib.MOVERS[mover], pieces=pieces, **core,
                                                             **kin)
    for k in _lib.EFFECTIVE_FIELDS:
        assert _bits(_np(r32[k])) == _bits(pieces[k]), k
    wd = dict(zip(("pressure", "temperature", "dewpoint") + WIND_KEYS, w32))
    bounds, excuse = _eff_bounds(want32, scale32, extra32, wd, True, _lib.MOVERS[mover])
    stat = _check_eff(r32, want32, bounds, excuse, f"{case}/row {row}/f32: ")
    print(f"REGIME_STAT arguments {case} row={row} {PAIRWISE[row]} near_threshold={near} jump_excused={jump} "
          f"f32_excused={max(e for e, _ in stat.values())}")


@pytest.mark.parametrize("arg", [(a, v) for a in ARG_NAMES for v in NON_DEFAULT[a]],
                         ids=[f"{a}={v}" for a in ARG_NAMES for v in NON_DEFAULT[a]])
def test_each_argument_changes_the_outputs(cache, arg):
    """An argument that is silently dropped leaves the outputs at the default run's: each must move some output on
    the argument cases' columns (and the outputs it cannot reach stay put)."""
    name, value = arg
    moved = {}
    for case in ARG_CASES:
        x = _arg_inputs(cache, case, np.float64, n=N_COLUMNS)
        ref = parcel.effective_layer_parameters(*x)
        got = parcel.effective_layer_parameters(*x, **{name: value})
        for k in ref:
            a, b = np.asarray(got[k]), np.asarray(ref[k])
            moved[k] = moved.get(k, 0) + int(((a != b) & ~(np.isnan(a) & np.isnan(b))).sum())
    assert sum(moved.values()) > 0, (name, value, moved)
    if name == "mixed_layer_depth":                   # the ML parcel only enters STP
        assert moved["significant_tornado_parameter"] > 0 and \
            all(v == 0 for k, v in moved.items() if k != "significant_tornado_parameter"), moved
    if name == "mover":                               # the same layer; the motion and the composites' sign change
        assert moved["effective_srh"] > 0 and moved["effective_inflow_base"] == 0, moved
    if name in ("min_cape", "min_cin"):
        assert moved["effective_inflow_base"] + moved["effective_inflow_top"] > 0, moved
    print(f"REGIME_STAT argument_moves {name}={value} {moved}")


# ---- 6. layouts ------------------------------------------------------------------------------------------------------------
LAYOUT_CASES = ("terrain_era5", "terrain")


@pytest.mark.parametrize("layout", ["NL", "4d", "L4d"])
@pytest.mark.parametrize("case", LAYOUT_CASES)
def test_layouts_give_the_same_bits(cache, case, layout):
    """effective_layer_parameters, bunkers_storm_motion and storm_relative_helicity on [N, L] (vert_axis=1), on
    (2, L, 25, 40) (vert_axis=1) and on (L, 2, 25, 40) (vert_axis=0) equal the [L, N] call bit for bit; on the ERA5
    case the pressure stays a shared 1-D axis."""
    assert N_COLUMNS == 2 * 25 * 40
    d = {k: v for k, v in cache.inputs(case).items() if k in ("pressure", "temperature", "dewpoint") + WIND_KEYS}
    L = d["temperature"].shape[0]
    mover = _mover(case)
    if layout == "L4d":
        lay = {k: (v if v.ndim == 1 and k == "pressure" else
                   v.reshape((2, 25, 40) if v.ndim == 1 else (L, 2, 25, 40))) for k, v in d.items()}
        va = 0
    else:
        lay, va = _to_layout(d, layout, L), 1

    def calls(x, vert_axis):
        e = parcel.effective_layer_parameters(*[x[k] for k in ("pressure", "temperature", "dewpoint") + WIND_KEYS],
                                              mover=mover, vert_axis=vert_axis)
        winds = [x[k] for k in ("surface_wind_u", "surface_wind_v", "wind_u", "wind_v", "wind_height_above_surface")]
        b = parcel.bunkers_storm_motion(*winds, vert_axis=vert_axis)
        s = parcel.storm_relative_helicity(*winds, depths=(500, 3000), mover=mover, vert_axis=vert_axis)
        return {**dict(e), **dict(b), **dict(s)}

    ref, got = calls(d, 0), calls(lay, va)
    assert set(got) == set(ref)
    for k in ref:
        g = np.asarray(got[k])
        assert g.shape == ((N_COLUMNS,) if layout == "NL" else (2, 25, 40)), (k, g.shape)
        assert _bits(np.asarray(ref[k])) == _bits(g.reshape(-1)), (case, layout, k)
    assert np.isfinite(np.asarray(ref["significant_tornado_parameter"])).mean() > 0.5


@pytest.mark.parametrize("case", LAYOUT_CASES)
def test_xarray_with_transposed_height(cache, case):
    """Through xarray DataArrays whose height has its dimensions in the other order than the winds (and the
    temperature): the layer aligns by name, so every output equals the NumPy [L, N] call bit for bit."""
    import xr_double
    d = {k: v for k, v in cache.inputs(case).items() if k in ("pressure", "temperature", "dewpoint") + WIND_KEYS}
    mover = _mover(case)
    ref_e = parcel.effective_layer_parameters(*[d[k] for k in ("pressure", "temperature", "dewpoint") + WIND_KEYS],
                                              mover=mover)
    winds = [d[k] for k in ("surface_wind_u", "surface_wind_v", "wind_u", "wind_v", "wind_height_above_surface")]
    ref_b = parcel.bunkers_storm_motion(*winds)
    ref_s = parcel.storm_relative_helicity(*winds, mover=mover)
    pf = xr_double.install()
    try:
        lv = "model_level_number"
        da = lambda a: xr_double.DataArray(a, dims=(lv, "x"))                # noqa: E731
        sa = lambda a: xr_double.DataArray(a, dims=("x",))                   # noqa: E731
        p = xr_double.DataArray(d["pressure"], dims=(lv,)) if d["pressure"].ndim == 1 else da(d["pressure"])
        h_t = xr_double.DataArray(np.ascontiguousarray(d["wind_height_above_surface"].T), dims=("x", lv))
        su, sv = sa(d["surface_wind_u"]), sa(d["surface_wind_v"])
        e = pf.effective_layer_parameters(p, da(d["temperature"]), da(d["dewpoint"]), h_t, da(d["wind_u"]),
                                          da(d["wind_v"]), su, sv, mover=mover)
        b = pf.bunkers_storm_motion(su, sv, da(d["wind_u"]), da(d["wind_v"]), h_t)
        s = pf.storm_relative_helicity(su, sv, da(d["wind_u"]), da(d["wind_v"]), h_t, mover=mover)
        for got, ref in ((e, ref_e), (b, ref_b), (s, ref_s)):
            assert set(got.keys()) == set(ref.keys())
            for k in ref:
                assert got[k].dims == ("x",), (k, got[k].dims)
                assert _bits(np.asarray(got[k].data)) == _bits(np.asarray(ref[k])), (case, k)
    finally:
        xr_double.uninstall()


# ---- 7. conv_properties(kinematics=True, effective=True) -----------------------------------------------------------------
CONV_N = 1000
CONV_VARIANTS = {"f64": (np.float64, False), "f32": (np.float32, False), "f32-cuda": (np.float32, True)}
CONV_PARAMS = [(c, v, m, False) for c in CONV_CASES for v in CONV_VARIANTS for m in ("right", "left")]
CONV_PARAMS += [("masked_era5", v, m, True) for v in CONV_VARIANTS for m in ("right", "left")]
NEW_FIELDS = list(_lib.MOTION_FIELDS) + ["srh_0_1000m", "srh_0_3000m"] + list(_lib.EFFECTIVE_PARAMETER_FIELDS)


def _conv_fields(cache, case):
    def make():
        regime, kw = CONV_CASES[case]
        i = list(CONV_CASES).index(case)
        p, t, td, p0 = rc.columns(regime, CONV_N, seed=1100 + i, **kw)
        return rc.conv_fields(p, t, td, p0, seed=1150 + i)
    return cache.get(("conv_fields", case), make)


def _conv_run(cache, case, variant, mover, ignore_nans):
    def make():
        ty, cuda = CONV_VARIANTS[variant]
        dat = {k: v.astype(ty) for k, v in _conv_fields(cache, case).items()}
        if cuda:
            dat = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in dat.items()}
        res = parcel.conv_properties(dat, ignore_nans=ignore_nans, metpy_compat=conv_compat(case), kinematics=True,
                                     effective=True, mover=mover)
        return dict(res), dat["dewpoint"]
    return cache.get(("conv_run", case, variant, mover, ignore_nans), make)


@pytest.mark.parametrize("param", CONV_PARAMS, ids=[f"{c}-{v}-{m}" + ("-ignore_nans" if i else "")
                                                     for c, v, m, i in CONV_PARAMS])
def test_conv_properties_kinematics_effective_against_oracle(ctx, cache, param):
    """The 12 kinematics / effective fields against the oracle's assembly: its conv_properties NaN mask (any NaN
    dewpoint from q, pressure, temperature or q in the column; none with ignore_nans), ko.storm_kinematics on the
    rounded winds and ko.effective_layer_parameters on the dewpoint the call derived, composed from the library's
    pieces.  NaN patterns exact; float32 CUDA tensors equal float32 NumPy bit for bit."""
    case, variant, mover, ignore_nans = param
    ty, _ = CONV_VARIANTS[variant]
    f32 = ty == np.float32
    compat = conv_compat(case)
    got, td = _conv_run(cache, case, variant, mover, ignore_nans)
    f = _conv_fields(cache, case)
    w = {k: v.astype(np.float64) for k, v in f.items()}
    P2 = np.broadcast_to(w["pressure"].reshape(w["pressure"].shape[0], -1), w["temperature"].shape)
    if ignore_nans:
        bad = np.zeros(CONV_N, dtype=bool)
    else:
        with np.errstate(all="ignore"):
            td_ora = th.dewpoint_from_specific_humidity(np.ascontiguousarray(P2), w["temperature"],
                                                        w["specific_humidity"], compat)
        bad = (np.isnan(td_ora) | np.isnan(P2) | np.isnan(w["temperature"]) |
               np.isnan(w["specific_humidity"])).any(axis=0)
        assert 0 < bad.sum() < CONV_N if case in ("masked_era5",) else bad.sum() < CONV_N
    want_k, scale_k = cache.get(("conv_kin", case, mover), lambda: ko.storm_kinematics(
        *[w[k] for k in WIND_KEYS], _lib.MOVERS[mover], (1000.0, 3000.0)))
    want_k = {k: np.where(bad, np.nan, v) for k, v in want_k.items()}
    kin_compare({k: got[k] for k in want_k}, want_k, scale_k, f32)
    # the effective-layer parameters on the dewpoint the call derived, composed from the library's pieces
    D = _np(td)
    pieces = cache.get(("conv_pieces", case, variant), lambda: _pieces(
        ctx, f["pressure"].astype(ty), f["temperature"].astype(ty), D.astype(ty), {"metpy_compat": compat}))
    want, scale, extra = ko.effective_layer_parameters(w["pressure"], w["temperature"], D, *[w[k] for k in WIND_KEYS],
                                                       cache.opts(compat), _lib.MOVERS[mover], pieces=pieces)
    bounds, excuse = _eff_bounds(want, scale, extra, w, f32, _lib.MOVERS[mover])
    for k in _lib.COMPOSITE_FIELDS:
        assert excuse[k].sum() <= JUMP_CAP * CONV_N, (k, int(excuse[k].sum()))
    stat = _check_eff(got, want, bounds, excuse, f"{param}: ", mask=bad)
    for k in NEW_FIELDS:
        assert np.isnan(_np(got[k])[bad]).all(), k
    if variant == "f32-cuda":
        other, _ = _conv_run(cache, case, "f32", mover, ignore_nans)
        for k in NEW_FIELDS:
            assert _bits(got[k]) == _bits(other[k]), k
    print(f"REGIME_STAT conv {case} {variant} {mover} ignore_nans={int(ignore_nans)} masked={int(bad.sum())} "
          + " ".join(f"{k}:excused={e},err/bound={q:.2g}" for k, (e, q) in stat.items()))
